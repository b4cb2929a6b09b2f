#!/usr/bin/env python
"""
Generate ``reference_classes.npz``: what the reference's own scorer / trainer / container classes pass to
``lenskit._accel`` and what they make of the answers, recorded with ``lenskit._accel`` bound to
``lkpy_b200.accel`` (INTEGRATION.md §1) and the device part of its entry points replaced by the CPU oracle.

    python tests/golden/make_reference_classes.py <lenskit source checkout>

Nothing at test time loads the reference: ``tests/test_reference_classes.py`` replays each record through this
package.  Arrays a test can rebuild from ``ml_small.npz`` with this package's own code (interaction matrices,
the seeded initial factors, the similarity matrix) are stored as digests, the rest as values.
"""

from __future__ import annotations

import ast
import sys
import warnings
from pathlib import Path

import numpy as np
import pytest

OUT = Path(__file__).resolve().parent
sys.path[:0] = [str(OUT), str(OUT.parent), str(OUT.parent.parent)]

import ref_sandbox  # noqa: E402
from helpers import TaskProbe, csr_digest, oracle_accel, sha256  # noqa: E402

from lkpy_b200 import accel, data  # noqa: E402

rec: dict[str, np.ndarray] = {}


def put(key: str, v) -> None:
    assert key not in rec, key
    rec[key] = np.asarray(v)


def arrow_type(a) -> str:
    """The Arrow storage type of a matrix argument (extension arrays are described by their storage)."""
    t = a.type
    return str(t.storage_type if hasattr(t, "storage_type") else t)


def put_matrix(key: str, m) -> None:
    csr = accel.as_host_csr(m)
    put(f"{key}.digest", csr_digest(csr))
    put(f"{key}.shape", csr.shape)
    put(f"{key}.arrow_type", arrow_type(m))


def put_arrow(key: str, a) -> None:
    """A small nullable Arrow array: values (nulls as 0 / NaN) and validity."""
    import pyarrow as pa

    a = a.combine_chunks() if isinstance(a, pa.ChunkedArray) else a
    put(f"{key}.type", str(a.type))
    put(f"{key}.valid", ~np.asarray(a.is_null().to_numpy(zero_copy_only=False)))
    fill = 0 if pa.types.is_integer(a.type) else np.nan
    put(f"{key}.values", np.asarray(a.fill_null(fill).to_numpy(zero_copy_only=False)))


class Recorder:
    """Wraps the entry points of ``lenskit._accel`` the reference calls; arguments are recorded at call time."""

    def __init__(self, mp):
        self.calls: list[tuple[str, tuple]] = []
        for ns, names in (
            (accel.als, ("train_implicit_matrix", "train_explicit_matrix")),
            (accel.knn, ("compute_similarities", "score_explicit", "score_implicit", "user_score_items_explicit",
                         "user_score_items_implicit")),
        ):  # fmt: skip
            for name in names:
                mp.setattr(ns, name, self._wrap(name, getattr(ns, name)))

    def _wrap(self, name, fn):
        def call(*args):
            snap = tuple(np.array(a) if isinstance(a, np.ndarray) else a for a in args)
            out = fn(*args)
            self.calls.append((name, snap, out))
            return out

        return call

    def take(self):
        calls, self.calls = self.calls, []
        return calls


def record_als(tag, calls, factors):
    """ALS half-steps: which matrix, which factor table is `this`, the Gram or scalar `reg` the reference passed."""
    put(f"{tag}/n_calls", len(calls))
    _name, (_m, this, other, _x), _t = calls[0]  # the user half comes first: the factors as initialised
    put(f"{tag}/init_user_digest", sha256(this))
    put(f"{tag}/init_item_digest", sha256(other))
    for i, (name, (matrix, this, other, extra), _task) in enumerate(calls):
        put(f"{tag}/call{i}.fn", name)
        put_matrix(f"{tag}/call{i}.matrix", matrix)
        put(f"{tag}/call{i}.this", "user" if this.shape[0] == factors[0].shape[0] else "item")
        put(f"{tag}/call{i}.extra", extra)  # OtOr (implicit) or reg (explicit)


def implicit_mf(ref, ml):
    imp, training = ref["lenskit.als._implicit"], ref["lenskit.training"]
    k, epochs = 16, 2
    m = imp.ImplicitMFScorer(embedding_size=k, epochs=epochs, regularization=0.1, weight=40)
    trainer = m.create_trainer(ref_sandbox.FakeDataset(ml), training.TrainingOptions(rng=42))
    metrics = [trainer.train_epoch() for _ in range(epochs)]
    put("implicit_mf/metric_names", sorted(metrics[0]))
    trainer.finalize()
    record_als("implicit_mf", REC.take(), (m.user_embeddings, m.item_embeddings))
    put("implicit_mf/user_embeddings", m.user_embeddings)
    put("implicit_mf/item_rows", ITEM_ROWS)
    put("implicit_mf/item_embeddings", m.item_embeddings[ITEM_ROWS])
    put("implicit_mf/otor_after_training", m._OtOr)


def implicit_mf_scores(ref, ml):
    imp, training, items_mod = ref["lenskit.als._implicit"], ref["lenskit.training"], ref["lenskit.data._items"]
    m = imp.ImplicitMFScorer(embedding_size=8, epochs=1, regularization=0.1, weight=40)
    m.train(ref_sandbox.FakeDataset(ml), training.TrainingOptions(rng=7))
    record_als("implicit_mf_scores", REC.take(), (m.user_embeddings, m.item_embeddings))
    tgt = np.array([0, 10, 200, 4000])
    out = m(ml.user_ids[5], items_mod.ItemList(item_ids=ml.item_ids[tgt]))
    put("implicit_mf_scores/user", 5)
    put("implicit_mf_scores/items", tgt)
    put("implicit_mf_scores/scores", out.scores("numpy"))


def biased_mf(ref, ml):
    exp, training, items_mod = ref["lenskit.als._explicit"], ref["lenskit.training"], ref["lenskit.data._items"]
    m = exp.BiasedMFScorer(embedding_size=8, epochs=2, regularization=0.1, damping=5.0)
    trainer = m.create_trainer(ref_sandbox.FakeDataset(ml), training.TrainingOptions(rng=3))
    for _ in range(2):
        trainer.train_epoch()
    trainer.finalize()
    record_als("biased_mf", REC.take(), (m.user_embeddings, m.item_embeddings))
    # the residuals after the reference's bias model: this package has no bias model to rebuild them with
    ui = accel.as_host_csr(trainer.ui_rates)
    put("biased_mf/ui_values", ui.values)
    put("biased_mf/user_embeddings", m.user_embeddings)
    put("biased_mf/item_rows", ITEM_ROWS)
    put("biased_mf/item_embeddings", m.item_embeddings[ITEM_ROWS])
    out = m(ml.user_ids[3], items_mod.ItemList(item_ids=ml.item_ids[[1, 50, 900]]))
    put("biased_mf/scores", out.scores("numpy"))


def item_knn(ref, ml):
    knn, training = ref["lenskit.knn.item"], ref["lenskit.training"]
    m = knn.ItemKNNScorer(max_nbrs=20, min_sim=1e-6, save_nbrs=20)
    m.train(ref_sandbox.FakeDataset(ml), training.TrainingOptions())
    ((name, (ui, iu, shape, min_sim, save_nbrs), _task),) = REC.take()
    put("item_knn/fn", name)
    put_matrix("item_knn/ui", ui)
    put_matrix("item_knn/iu", iu)
    put("item_knn/shape", shape)
    put("item_knn/min_sim", min_sim)
    put("item_knn/save_nbrs", save_nbrs)
    sim = m.sim_matrix
    put("item_knn/sim_extension", sim.type.extension_name)
    put("item_knn/sim_dimension", sim.type.dimension)
    put_matrix("item_knn/sim", sim)
    put("item_knn/item_means", np.asarray(m.item_means, dtype=np.float32))
    put("item_knn/item_counts", np.asarray(m.item_counts))


def item_knn_scores(ref, ml, feedback):
    knn, training, items_mod = ref["lenskit.knn.item"], ref["lenskit.training"], ref["lenskit.data._items"]
    ItemList = items_mod.ItemList
    m = knn.ItemKNNScorer(max_nbrs=20, min_sim=1e-6, save_nbrs=20, feedback=feedback)
    m.train(ref_sandbox.FakeDataset(ml), training.TrainingOptions())
    REC.take()
    accel.clear_cache()
    R = ml.coo().tocsr()
    u = int(np.argmax(np.diff(R.indptr)))
    nums = R.indices[R.indptr[u] : R.indptr[u + 1]]
    rates = R.data[R.indptr[u] : R.indptr[u + 1]].astype(np.float32)
    unknown = int(ml.item_ids.max()) + 1000
    hist = ItemList(item_ids=np.concatenate([ml.item_ids[nums], [unknown]]), rating=np.concatenate([rates, [3.0]]))
    tgt_nums = np.arange(0, ml.n_items, 7)
    targets = ItemList(item_ids=np.concatenate([ml.item_ids[tgt_nums], [unknown + 1]]))
    out = m(hist, targets)
    ((name, args, (scores, counts)),) = REC.take()
    t = f"item_knn_{feedback}"
    put(f"{t}/fn", name)
    put_matrix(f"{t}/sims", args[0])
    for nm, a in zip(("ref_items", "ref_rates", "tgt_items") if len(args) == 6 else ("ref_items", "tgt_items"), args[1:-2]):
        put_arrow(f"{t}/{nm}", a)
    put(f"{t}/max_nbrs", args[-2])
    put(f"{t}/min_nbrs", args[-1])
    put_arrow(f"{t}/ret_scores", scores)
    put_arrow(f"{t}/ret_counts", counts)
    put(f"{t}/scores", out.scores("numpy"))
    put(f"{t}/nbr_counts", np.asarray(out.field("nbr_counts", "numpy"), dtype=np.float64))


def user_knn_scores(ref, ml, feedback):
    usr, training, items_mod = ref["lenskit.knn.user"], ref["lenskit.training"], ref["lenskit.data._items"]
    m = usr.UserKNNScorer(max_nbrs=15, min_nbrs=2, min_sim=1e-6, feedback=feedback)
    m.train(ref_sandbox.FakeDataset(ml), training.TrainingOptions())
    accel.clear_cache()
    tgt = np.arange(0, ml.n_items, 11)
    out = m(ml.user_ids[42], items_mod.ItemList(item_ids=ml.item_ids[tgt]))
    ((name, (tgt_items, nbr_rows, nbr_sims, ratings, max_nbrs, min_nbrs), ret),) = REC.take()
    t = f"user_knn_{feedback}"
    put(f"{t}/fn", name)
    put_arrow(f"{t}/tgt_items", tgt_items)
    put_arrow(f"{t}/nbr_rows", nbr_rows)
    put_arrow(f"{t}/nbr_sims", nbr_sims)
    put_matrix(f"{t}/ratings", ratings)
    r = accel.as_host_csr(ratings)
    if feedback == "explicit":  # user-centred ratings
        put(f"{t}/ratings_values", r.values)
    put(f"{t}/max_nbrs", max_nbrs)
    put(f"{t}/min_nbrs", min_nbrs)
    put_arrow(f"{t}/ret_scores", ret)
    put(f"{t}/scores", out.scores("numpy"))


def index_type(ref):
    """The reference's ``SparseIndexType`` and the row type ``SparseRowArray.from_array`` gives this package's
    result chunks, as an Arrow IPC stream (extension names and metadata travel in the schema)."""
    import pyarrow as pa

    matrix = ref["lenskit.data.matrix"]
    t = matrix.SparseIndexType(77)
    put("index_type/extension_name", t.extension_name)
    put("index_type/serialized", np.frombuffer(t.__arrow_ext_serialize__(), dtype=np.uint8))
    put("index_type/storage", str(t.storage_type))
    csr = data.InteractionCSR(np.array([0, 2, 2, 3], np.int64), np.array([1, 5, 0], np.int32),
                              np.array([0.5, 0.25, 1.0], np.float32), (3, 77))  # fmt: skip
    arr = pa.chunked_array(accel.csr_to_arrow_chunks(csr, 2)).combine_chunks()
    wrapped = matrix.SparseRowArray.from_array(arr)
    assert wrapped.shape == (3, 77)
    sink = pa.BufferOutputStream()
    tbl = pa.table({"rows": wrapped})
    with pa.ipc.new_stream(sink, tbl.schema) as w:
        w.write_table(tbl)
    put("index_type/wrapped_ipc", np.frombuffer(sink.getvalue().to_pybytes(), dtype=np.uint8))


def task_runner(_ref):
    import sys

    run = sys.modules["lenskit.parallel"].run_accel_task
    prog = ref_sandbox._Progress()
    ok = TaskProbe(42.0)
    assert run(ok, progress=prog) == 42.0 and prog.updates >= 1
    put("task_runner/ok_log", ok.log)
    bad = TaskProbe(error=RuntimeError("ALS solve error: array minor of row 3 is not positive"))
    with pytest.raises(RuntimeError) as ei:
        run(bad)
    assert ei.value.__cause__ is bad.error
    put("task_runner/error_message", str(ei.value))
    put("task_runner/error_log", bad.log)


def top_n(ref):
    ItemList = ref["lenskit.data._items"].ItemList
    rng = np.random.default_rng(8)
    scores = rng.standard_normal(200).astype(np.float32)
    scores[::9] = np.nan
    seen = []
    real = accel.argtopn

    def spy(s, n):
        out = real(s, n)
        seen.append((s, n, out))
        return out

    sys.modules["lenskit._accel"].data.argtopn = spy
    top = ItemList(item_ids=np.arange(1000, 1200), scores=scores).top_n(10)
    sys.modules["lenskit._accel"].data.argtopn = real
    ((s, n, out),) = seen
    put_arrow("top_n/arg", s)
    put("top_n/n", n)
    put("top_n/ids", top.ids())
    put("top_n/ordered", top.ordered)


def trainer_api(ref):
    """What INTEGRATION.md's trainer binding relies on: the fields of ``TrainContext`` and the methods of the
    classes it subclasses."""
    imp, common = ref["lenskit.als._implicit"], ref["lenskit.als._common"]
    put("trainer_api/context_fields", list(common.TrainContext._fields))
    for cls in (imp.ImplicitMFTrainer, imp.ImplicitMFScorer):
        put(f"trainer_api/{cls.__name__}.methods", sorted(n for n in dir(cls) if callable(getattr(cls, n, None))))
        put(f"trainer_api/{cls.__name__}.abstract", sorted(getattr(cls, "__abstractmethods__", ())))


def stub_signatures(root: Path):
    """Parameter names, in order, of every function the typed stubs ``_accel/als.pyi`` and ``_accel/knn.pyi``
    declare: the reference's call sites bind them positionally."""
    for mod in ("als", "knn"):
        tree = ast.parse((root / "src" / "lenskit" / "_accel" / f"{mod}.pyi").read_text())
        fns = [n for n in tree.body if isinstance(n, ast.FunctionDef)]
        put(f"stubs/{mod}", [fn.name for fn in fns])
        for fn in fns:
            put(f"stubs/{mod}.{fn.name}", [a.arg for a in fn.args.args])


if __name__ == "__main__":
    ref_sandbox.set_root(Path(sys.argv[1]))
    ml = data.load_ml_small()
    ITEM_ROWS = np.sort(np.random.default_rng(0).choice(ml.n_items, 1024, replace=False))
    with ref_sandbox.reference_modules() as ref, warnings.catch_warnings(), pytest.MonkeyPatch.context() as mp:
        warnings.simplefilter("ignore")  # "not the short import path": the sandbox has no lenskit/__init__
        oracle_accel(mp)
        REC = Recorder(mp)
        implicit_mf(ref, ml)
        implicit_mf_scores(ref, ml)
        biased_mf(ref, ml)
        item_knn(ref, ml)
        for fb in ("explicit", "implicit"):
            item_knn_scores(ref, ml, fb)
            user_knn_scores(ref, ml, fb)
        index_type(ref)
        task_runner(ref)
        top_n(ref)
        trainer_api(ref)
    stub_signatures(Path(sys.argv[1]))
    np.savez_compressed(OUT / "reference_classes.npz", **rec)
    print((OUT / "reference_classes.npz").stat().st_size, "bytes,", len(rec), "arrays")
