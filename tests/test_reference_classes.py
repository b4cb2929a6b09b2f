"""
The function-level drop-in of INTEGRATION.md §1 as the reference's OWN classes use it: ``lenskit.training``,
``als._common`` / ``als._implicit`` / ``als._explicit``, ``knn.item`` / ``knn.user``, ``data.matrix.SparseRowArray``,
``ItemList`` and ``parallel._task.run_accel_task``, run with ``lenskit._accel`` bound to ``lkpy_b200.accel``, left a
record of every call they made into the accelerator API and of what they made of the answers
(``golden/reference_classes.npz``, written by ``golden/make_reference_classes.py``).  Each test replays one record
through this package: the same arguments in the same Arrow layouts, in the same order, and the answers must be
the ones the reference's classes received and built their models and scores from.

Inputs this package can rebuild from ``ml_small.npz`` (the interaction matrices, the seeded initial factors, the
similarity matrix) are rebuilt and checked against the recorded digests.  Without a CUDA device the device part
of the entry points is replaced by the oracle (``helpers.oracle_accel``); everything else — Arrow ingest, the
task protocol, the in-place contract on ``this``, the result layout — is the product code.
"""

import ast
import re
from pathlib import Path

import numpy as np
import pyarrow as pa
import pytest
import scipy.sparse as sps
import torch
from helpers import TaskProbe, csr_digest, explicit_init, implicit_init, oracle_accel, rel_fro, sha256

import oracle
from lkpy_b200 import accel, data

GOLD = Path(__file__).resolve().parent / "golden"
ON_GPU = torch.cuda.is_available()
TOL = 1e-4 if ON_GPU else 1e-6  # device arithmetic vs the oracle the record was made with
GRAM_TOL = 1e-4  # the reference's f32 OtOr against the oracle's: the same sums in another order


@pytest.fixture(scope="module")
def z():
    with np.load(GOLD / "reference_classes.npz") as f:
        return {k: f[k] for k in f.files}


@pytest.fixture(scope="module", autouse=True)
def device_part():
    with pytest.MonkeyPatch.context() as mp:
        if ON_GPU:
            from lkpy_b200 import _build

            _build.build()
        else:
            oracle_accel(mp)
        yield


def s(z, key) -> str:
    return str(z[key])


def rows_arrow(csr: data.InteractionCSR, arrow_type: str, structure_only: bool = False):
    """A sparse row matrix in the Arrow storage layout the reference's ``SparseRowArray`` passed (List or
    LargeList of Struct{index: lenskit.sparse_index, value: float32}, or of the bare index)."""
    idx = pa.ExtensionArray.from_storage(accel.sparse_index_type(csr.shape[1]), pa.array(csr.indices, type=pa.int32()))
    elems = idx if structure_only else pa.StructArray.from_arrays([idx, pa.array(csr.values, type=pa.float32())],
                                                                 names=["index", "value"])  # fmt: skip
    large = arrow_type.startswith("large_list")
    offs = pa.array(np.asarray(csr.indptr, dtype=np.int64 if large else np.int32))
    arr = (pa.LargeListArray if large else pa.ListArray).from_arrays(offs, elems)
    assert str(arr.type) == arrow_type
    return arr


def recorded_matrix(z, key, csr, structure_only=False):
    """``csr`` rebuilt by this package, checked against the digest of what the reference passed under ``key``."""
    assert csr_digest(csr) == s(z, f"{key}.digest"), f"{key}: rebuilt matrix differs from the recorded one"
    return rows_arrow(csr, s(z, f"{key}.arrow_type"), structure_only)


def recorded_arrow(z, key):
    t = {"int32": pa.int32(), "float": pa.float32()}[s(z, f"{key}.type")]
    return pa.array(z[f"{key}.values"], type=t, mask=~z[f"{key}.valid"])


def assert_same_arrow(got, z, key):
    """Equal to the recorded answer: type, nulls, and value bits."""
    got = got.combine_chunks() if isinstance(got, pa.ChunkedArray) else got
    assert str(got.type) == s(z, f"{key}.type")
    valid = ~np.asarray(got.is_null().to_numpy(zero_copy_only=False))
    assert np.array_equal(valid, z[f"{key}.valid"])
    g = np.asarray(got.fill_null(0).to_numpy(zero_copy_only=False))
    assert np.array_equal(g[valid].view(np.int32), z[f"{key}.values"][valid].view(np.int32))


def replay_als(z, tag, mats, csrs, tables) -> float:
    """The recorded half-steps, in order, on the same matrices and factor tables; returns the tolerance of the
    final factors against the recorded ones.  Without a device the oracle replays the record exactly.  On the
    device each half-step meets the bar of test_als_gpu.py against the f64 oracle of that step: 1e-4 where f32
    arithmetic can deliver it, else no worse than the f32 oracle (the reference init makes the early
    ml-latest-small systems that ill-conditioned).  The recorded chain and the device's may each carry that
    f32 error at every step, in opposite directions."""
    tol = TOL
    for i in range(int(z[f"{tag}/n_calls"])):
        fn = s(z, f"{tag}/call{i}.fn")
        this_name = s(z, f"{tag}/call{i}.this")
        other_name = "item" if this_name == "user" else "user"
        this, other, extra = tables[this_name], tables[other_name], z[f"{tag}/call{i}.extra"]
        mode = "implicit" if fn == "train_implicit_matrix" else "explicit"
        o32, o64 = oracle.otor(other, 0.1)
        if mode == "implicit":
            # the Gram the reference hands over: OtOr + reg I of the other side it holds (_implicit_otor); on the
            # device the factors leave the record's after the first half-step, and the Gram is that of the
            # factors held here
            if i == 0 or not ON_GPU:
                assert rel_fro(extra, o32) < GRAM_TOL
            arg = o32 if ON_GPU else extra
        else:
            arg = float(extra)
        if ON_GPU:
            kw = dict(otor_mat=o64) if mode == "implicit" else dict(reg=arg)
            ref64, _ = oracle.als_half_f64(mode, csrs[this_name], this, other, **kw)
            kw = dict(otor_mat=o32) if mode == "implicit" else dict(reg=arg)
            ref32, _ = oracle.als_half(mode, csrs[this_name], this, other, **kw)
            e_cpu = rel_fro(ref32, ref64)
        train = accel.als.train_implicit_matrix if mode == "implicit" else accel.als.train_explicit_matrix
        delta = accel.run_accel_task(train(mats[this_name], this, other, arg))
        assert np.isfinite(delta) and delta > 0
        assert tables[this_name] is this  # updated in place (TrainContext.left)
        if ON_GPU:
            e_gpu = rel_fro(this, ref64)
            assert e_gpu <= (TOL if e_cpu <= TOL / 3 else 1.5 * e_cpu + 2e-6), (i, e_gpu, e_cpu)
            tol += 2 * e_cpu
    return tol


def test_reference_implicit_mf_trains_through_the_shim(z, ml_small):
    """``ImplicitMFScorer.train`` (training.py:301-334 -> als/_common.py:209-256 -> als/_implicit.py:158-164):
    R and Rᵀ as SparseRowArrays, the factors initialised items first, ``als.train_implicit_matrix`` once per
    half-epoch.  Replayed here, the factors end where the reference's trainer left them."""
    tag = "implicit_mf"
    ui, iu = data.als_implicit_matrices(ml_small, 40.0)
    p, q = implicit_init(np.random.default_rng(42), ml_small.n_items, ml_small.n_users, 16)
    assert sha256(p) == s(z, f"{tag}/init_user_digest") and sha256(q) == s(z, f"{tag}/init_item_digest")
    mats = {"user": recorded_matrix(z, f"{tag}/call0.matrix", ui), "item": recorded_matrix(z, f"{tag}/call1.matrix", iu)}
    assert [s(z, f"{tag}/call{i}.this") for i in range(4)] == ["user", "item"] * 2
    assert list(z[f"{tag}/metric_names"]) == ["deltaP", "deltaQ"]
    tol = replay_als(z, tag, mats, {"user": ui, "item": iu}, {"user": p, "item": q})
    assert rel_fro(p, z[f"{tag}/user_embeddings"]) <= tol
    assert rel_fro(q[z[f"{tag}/item_rows"]], z[f"{tag}/item_embeddings"]) <= tol
    assert rel_fro(oracle.otor(q, 0.1)[0], z[f"{tag}/otor_after_training"]) <= GRAM_TOL + 2 * tol


def test_reference_item_knn_trains_through_the_shim(z, ml_small):
    """``ItemKNNScorer.train`` (knn/item.py:121-199): the reference centres and normalises, hands two
    SparseRowArrays to ``knn.compute_similarities``, concatenates the returned chunks and wraps them with
    ``SparseRowArray.from_array`` — which only accepts an index field of the ``lenskit.sparse_index``
    extension type (data/matrix.py:530-546).  The replayed call returns the recorded model, bit for bit."""
    ui, iu, means = data.knn_item_matrices(ml_small, True)
    assert s(z, "item_knn/fn") == "compute_similarities"
    shape, min_sim, save_nbrs = tuple(int(v) for v in z["item_knn/shape"]), float(z["item_knn/min_sim"]), int(z["item_knn/save_nbrs"])
    assert shape == (ml_small.n_users, ml_small.n_items)
    task = accel.knn.compute_similarities(recorded_matrix(z, "item_knn/ui", ui), recorded_matrix(z, "item_knn/iu", iu),
                                          shape, min_sim, save_nbrs)  # fmt: skip
    sim = pa.chunked_array(accel.run_accel_task(task)).combine_chunks()
    assert str(sim.type) == s(z, "item_knn/sim.arrow_type")
    assert sim.type.value_type.field("index").type.dimension == int(z["item_knn/sim_dimension"]) == ml_small.n_items
    got = accel.as_host_csr(sim, ml_small.n_items)
    assert csr_digest(got) == s(z, "item_knn/sim.digest")
    want = oracle.knn_build(ui, iu, min_sim, save_nbrs)
    assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.values.view(np.int32), want.data.view(np.int32))
    assert np.array_equal(z["item_knn/item_means"].view(np.int32), means.view(np.int32))
    assert np.array_equal(z["item_knn/item_counts"], np.diff(got.indptr))


def test_result_index_field_is_the_reference_extension_type(z):
    """Wire format of the ``index`` field: extension name, JSON metadata and storage of the reference's
    ``SparseIndexType`` (data/matrix.py:104-146).  The reference wrapped this package's result chunks in its
    ``SparseRowArray`` and wrote them through Arrow IPC; that stream reads back here to the same CSR, and its
    ``index`` field carries the metadata this package writes."""
    t = accel.sparse_index_type(77)
    assert t.extension_name == s(z, "index_type/extension_name") and t.dimension == 77
    assert t.__arrow_ext_serialize__() == z["index_type/serialized"].tobytes()
    assert str(t.storage_type) == s(z, "index_type/storage")
    csr = data.InteractionCSR(np.array([0, 2, 2, 3], np.int64), np.array([1, 5, 0], np.int32),
                              np.array([0.5, 0.25, 1.0], np.float32), (3, 77))  # fmt: skip
    ours = pa.chunked_array(accel.csr_to_arrow_chunks(csr, 2)).combine_chunks()

    def ipc(tbl):
        sink = pa.BufferOutputStream()
        with pa.ipc.new_stream(sink, tbl.schema) as w:
            w.write_table(tbl)
        return pa.ipc.open_stream(sink.getvalue()).read_all()

    theirs = pa.ipc.open_stream(pa.py_buffer(z["index_type/wrapped_ipc"].tobytes())).read_all()
    mine = ipc(pa.table({"rows": ours}))

    def index_meta(tbl):
        return tbl.schema.field("rows").type.value_type.field("index").metadata

    assert index_meta(theirs) == index_meta(mine)
    assert index_meta(mine)[b"ARROW:extension:name"] == b"lenskit.sparse_index"
    back = accel.as_host_csr(theirs.column("rows").combine_chunks(), 77)
    assert back.shape == (3, 77) and np.array_equal(back.indptr, csr.indptr)
    assert np.array_equal(back.indices, csr.indices) and np.array_equal(back.values, csr.values)


@pytest.mark.parametrize("feedback", ["explicit", "implicit"])
def test_reference_item_knn_scores_through_the_shim(z, ml_small, feedback):
    """``ItemKNNScorer.__call__`` (knn/item.py:230-295) with the reference's real ``ItemList`` / ``Vocabulary``:
    nullable Int32 / Float32 Arrow arrays in (unknown history items and unknown targets are nulls), nullable
    score and count arrays out, the means added back by the reference.  The replayed call answers what the
    reference received, bit for bit, and that equals the oracle's accumulator."""
    t = f"item_knn_{feedback}"
    explicit = feedback == "explicit"
    assert s(z, f"{t}/fn") == ("score_explicit" if explicit else "score_implicit")
    ui, iu, means = data.knn_item_matrices(ml_small, explicit)
    S = oracle.knn_build(ui, iu, 1e-6, 20)
    sims = recorded_matrix(z, f"{t}/sims", data.InteractionCSR(S.indptr.astype(np.int64), S.indices, S.data, S.shape))
    names = ("ref_items", "ref_rates", "tgt_items") if explicit else ("ref_items", "tgt_items")
    args = [recorded_arrow(z, f"{t}/{n}") for n in names]
    max_nbrs, min_nbrs = int(z[f"{t}/max_nbrs"]), int(z[f"{t}/min_nbrs"])
    accel.clear_cache()
    fn = accel.knn.score_explicit if explicit else accel.knn.score_implicit
    scores, counts = fn(sims, *args, max_nbrs, min_nbrs)
    assert_same_arrow(scores, z, f"{t}/ret_scores")
    assert_same_arrow(counts, z, f"{t}/ret_counts")

    ri, ti = (np.asarray(a.fill_null(-1).to_numpy(zero_copy_only=False)) for a in (args[0], args[-1]))
    rv = None
    if explicit:
        rv = np.asarray(args[1].fill_null(np.nan).to_numpy(zero_copy_only=False), dtype=np.float32)[ri >= 0]
    want, want_ct = oracle.knn_score(S, ri[ri >= 0].astype(np.int32), rv, ti[ti >= 0].astype(np.int32), max_nbrs, min_nbrs)
    final = z[f"{t}/scores"]
    ok = ~np.isnan(want)
    assert ok.sum() > 100 and np.array_equal(np.isnan(final[ti >= 0]), ~ok) and np.isnan(final[ti < 0]).all()
    if explicit:
        want = want + means[ti[ti >= 0]]
    assert np.array_equal(want[ok].astype(np.float32).view(np.int32), final[ti >= 0][ok].astype(np.float32).view(np.int32))
    assert np.array_equal(z[f"{t}/nbr_counts"][ti >= 0][ok], want_ct[ok].astype(np.float64))


def test_reference_implicit_mf_scores_after_training_through_the_shim(z, ml_small):
    """The model the reference's trainer leaves behind is the one its own ``ALSBase.__call__`` scores with
    (als/_common.py:133-175): known user -> P[u] . Q^T over the requested items.  The replayed epoch gives the
    reference's scores."""
    tag = "implicit_mf_scores"
    ui, iu = data.als_implicit_matrices(ml_small, 40.0)
    p, q = implicit_init(np.random.default_rng(7), ml_small.n_items, ml_small.n_users, 8)
    assert sha256(p) == s(z, f"{tag}/init_user_digest") and sha256(q) == s(z, f"{tag}/init_item_digest")
    mats = {"user": recorded_matrix(z, f"{tag}/call0.matrix", ui), "item": recorded_matrix(z, f"{tag}/call1.matrix", iu)}
    tol = replay_als(z, tag, mats, {"user": ui, "item": iu}, {"user": p, "item": q})
    got = q[z[f"{tag}/items"]] @ p[int(z[f"{tag}/user"])]
    want = z[f"{tag}/scores"]
    assert np.allclose(got, want, rtol=10 * tol, atol=tol * np.abs(want).max())


def test_reference_biased_mf_trains_through_the_shim(z, ml_small):
    """``BiasedMFScorer`` (als/_explicit.py:94-118): the reference learns its bias model, builds the residual
    matrices and calls ``als.train_explicit_matrix(matrix, this, other, reg)`` — the scalar ``reg`` (scaled by
    the row's nnz inside, explicit.rs:104-108) instead of a Gram.  The residuals are recorded; replayed on
    them, the factors end where the reference's trainer left them."""
    tag = "biased_mf"
    R = sps.csr_array(ml_small.coo().tocsr())
    R.sort_indices()
    R.data = z[f"{tag}/ui_values"]
    ui = data.InteractionCSR.from_scipy(R)
    iu = data.InteractionCSR.from_scipy(R.T)
    p, q = explicit_init(np.random.default_rng(3), ml_small.n_items, ml_small.n_users, 8)
    assert sha256(p) == s(z, f"{tag}/init_user_digest") and sha256(q) == s(z, f"{tag}/init_item_digest")
    mats = {"user": recorded_matrix(z, f"{tag}/call0.matrix", ui), "item": recorded_matrix(z, f"{tag}/call1.matrix", iu)}
    assert {s(z, f"{tag}/call{i}.fn") for i in range(4)} == {"train_explicit_matrix"}
    tol = replay_als(z, tag, mats, {"user": ui, "item": iu}, {"user": p, "item": q})
    assert rel_fro(p, z[f"{tag}/user_embeddings"]) <= tol
    assert rel_fro(q[z[f"{tag}/item_rows"]], z[f"{tag}/item_embeddings"]) <= tol
    assert np.all(np.isfinite(z[f"{tag}/scores"]))


@pytest.mark.parametrize("feedback", ["explicit", "implicit"])
def test_reference_user_knn_scores_through_the_shim(z, ml_small, feedback):
    """``UserKNNScorer.__call__`` (knn/user.py:157-255) -> ``knn.user_score_items_explicit / _implicit``
    (user_score.rs:21-98): the neighbour list (Int32 rows, Float32 similarities) and the reference's own
    ``user_ratings`` SparseRowArray go in, a nullable Float32 array comes out, the user mean is added by the
    reference.  The replayed call answers what the reference received, which is the oracle's accumulator."""
    t = f"user_knn_{feedback}"
    explicit = feedback == "explicit"
    assert s(z, f"{t}/fn") == f"user_score_items_{feedback}"
    R = sps.csr_array(ml_small.coo().tocsr())
    R.sort_indices()
    R.data = z[f"{t}/ratings_values"] if explicit else np.ones(R.nnz, np.float32)  # user-centred ratings / structure
    rat = data.InteractionCSR.from_scipy(R)
    ratings = recorded_matrix(z, f"{t}/ratings", rat, structure_only=not explicit)
    tgt, rows, sims = (recorded_arrow(z, f"{t}/{n}") for n in ("tgt_items", "nbr_rows", "nbr_sims"))
    max_nbrs, min_nbrs = int(z[f"{t}/max_nbrs"]), int(z[f"{t}/min_nbrs"])
    accel.clear_cache()
    fn = accel.knn.user_score_items_explicit if explicit else accel.knn.user_score_items_implicit
    got = fn(tgt, rows, sims, ratings, max_nbrs, min_nbrs)
    assert_same_arrow(got, z, f"{t}/ret_scores")
    want, _ct = oracle.user_score(R, rows.to_numpy(), sims.to_numpy(), tgt.to_numpy(), max_nbrs, min_nbrs, explicit=explicit)
    ok = ~np.isnan(want)
    assert ok.sum() > 50 and np.array_equal(np.isnan(z[f"{t}/scores"]), ~ok)
    assert np.array_equal(want[ok].view(np.int32), z[f"{t}/ret_scores.values"][ok].view(np.int32))


def test_reference_task_runner_drives_the_task_mirror(z):
    """``run_accel_task`` (parallel/_task.py:25-57) asks a task for exactly this: ``invoke(pool=None)`` on an
    ``AccelTask-*`` worker thread, ``current_progress()`` polls while a progress object is given, failures
    re-raised as its RuntimeError with the task's exception as the cause.  The mirror asks the same of a
    probe task, and this package's ``AccelTask`` answers it: result hand-back, progress tuples, failures and
    cancellation."""
    import threading
    import time

    probe = TaskProbe(42.0)
    assert accel.run_accel_task(probe, progress=type("P", (), {"update": lambda *_a, **_k: None})()) == 42.0
    assert probe.log == list(z["task_runner/ok_log"])
    bad = TaskProbe(error=RuntimeError("ALS solve error: array minor of row 3 is not positive"))
    with pytest.raises(RuntimeError) as ei:
        accel.run_accel_task(bad)
    assert str(ei.value) == s(z, "task_runner/error_message") and ei.value.__cause__ is bad.error
    assert bad.log == list(z["task_runner/error_log"])

    seen = {}

    def body(task):
        seen["thread"] = threading.current_thread().name
        time.sleep(0.5)
        return 42.0

    updates = []
    prog = type("P", (), {"update": lambda _s, **kw: updates.append(kw)})()
    assert accel.run_accel_task(accel.AccelTask(body, total=10), progress=prog) == 42.0
    assert seen["thread"].startswith("AccelTask") and updates and all(set(u) == {"completed", "total"} for u in updates)

    def boom(_task):
        raise RuntimeError("ALS solve error: array minor of row 3 is not positive")

    with pytest.raises(RuntimeError, match="accelerator task failed") as ei:
        accel.run_accel_task(accel.AccelTask(boom, total=1))
    assert "ALS solve error" in str(ei.value.__cause__)
    t = accel.AccelTask(body, total=1)
    t.cancel()
    with pytest.raises(RuntimeError, match="accelerator task failed") as ei:
        accel.run_accel_task(t)
    assert "cancelled" in str(ei.value.__cause__)


def test_reference_item_list_top_n_through_the_argtopn_mirror(z):
    """``ItemList.top_n`` (data/_items.py:942-998) -> ``_accel.data.argtopn(scores: pa.Array, n)``: Arrow nulls
    and NaNs are both unscored (sorting.rs:163-167), an Int32Array of positions comes back, best first.  The
    replayed call picks the items the reference's list returned."""
    arg = recorded_arrow(z, "top_n/arg")
    got = accel.argtopn(arg, int(z["top_n/n"]))
    assert isinstance(got, pa.Array) and got.type == pa.int32()
    assert (1000 + got.to_numpy()).tolist() == z["top_n/ids"].tolist() and bool(z["top_n/ordered"])
    scores = arg.to_numpy(zero_copy_only=False)
    assert got.to_numpy().tolist() == oracle.argtopn(scores.astype(np.float32), 10).tolist()
    # nullable Arrow scores, as the kNN entry points return them
    masked = np.zeros(200, dtype=bool)
    masked[::4] = True
    got = accel.argtopn(pa.array(scores, mask=masked), 25)
    assert isinstance(got, pa.Array) and got.type == pa.int32()
    assert got.to_numpy().tolist() == oracle.argtopn(np.where(masked, np.nan, scores).astype(np.float32), 25).tolist()


def test_integration_md_trainer_binding_matches_both_sides(z):
    """The trainer-level binding printed in INTEGRATION.md §2 compiles; it subclasses the reference's
    ``ImplicitMFTrainer`` / ``ImplicitMFScorer`` (which leave no abstract method to fill) and overrides only
    methods they have; every ``engine.*`` / ``_lib.*`` name it uses exists in this package, and every
    ``context.*`` field it reads exists on the reference's ``TrainContext``."""
    from lkpy_b200 import _lib, engine

    text = (Path(__file__).resolve().parent.parent / "INTEGRATION.md").read_text()
    blocks = re.findall(r"```python\n(.*?)```", text, flags=re.S)
    block = next(b for b in blocks if "class B200ImplicitMFTrainer" in b)
    tree = ast.parse(block)
    compile(tree, "INTEGRATION.md#trainer-binding", "exec")
    imported = {a.name for n in ast.walk(tree) if isinstance(n, ast.ImportFrom) and n.module == "lenskit.als._implicit"
                for a in n.names}  # fmt: skip
    classes = {n.name: n for n in tree.body if isinstance(n, ast.ClassDef)}
    for ours, base in (("B200ImplicitMFTrainer", "ImplicitMFTrainer"), ("B200ImplicitMFScorer", "ImplicitMFScorer")):
        assert base in imported and [b.id for b in classes[ours].bases] == [base]
        assert list(z[f"trainer_api/{base}.abstract"]) == []
        methods = set(z[f"trainer_api/{base}.methods"])
        for fn in (n for n in classes[ours].body if isinstance(n, ast.FunctionDef)):
            assert not fn.decorator_list
            assert fn.name.startswith("_") or fn.name in methods, f"{ours}.{fn.name} overrides nothing of {base}"
    used = {(n.value.id, n.attr) for n in ast.walk(tree) if isinstance(n, ast.Attribute) and isinstance(n.value, ast.Name)}
    for mod_name, mod in (("engine", engine), ("_lib", _lib)):
        for _m, attr in sorted(u for u in used if u[0] == mod_name):
            assert hasattr(mod, attr), f"INTEGRATION.md uses {mod_name}.{attr}, which does not exist"
    fields = set(z["trainer_api/context_fields"])
    for _m, attr in sorted(u for u in used if u[0] in ("context", "ctx")):
        assert attr in fields, f"INTEGRATION.md reads context.{attr}; TrainContext has {sorted(fields)}"
