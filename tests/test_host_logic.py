"""
The roofline arithmetic of bench.py against the figures of SURVEY.md §8d (algorithmic bytes per
half-epoch / per build at ML-25M shape), and the host-side helpers that do not need a GPU.
"""

import importlib.util

import numpy as np
import pytest
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def _bench():
    spec = importlib.util.spec_from_file_location("lk_bench", ROOT / "bench.py")
    mod = importlib.util.module_from_spec(spec)
    sys.modules["lk_bench"] = mod
    spec.loader.exec_module(mod)
    return mod


def test_als_algorithmic_bytes_match_survey():
    b = _bench()
    U, I, N, k = 162_541, 59_047, 25_000_095, 64
    # SURVEY.md §8d: N(k s + 8) + 4(R+1) + R k 4 2 + k^2 4 per half-epoch (OtOr pass counted separately)
    fp32 = b.als_half_bytes(U, I, N, k, 4, False) + b.als_half_bytes(I, U, N, k, 4, False)
    bf16 = b.als_half_bytes(U, I, N, k, 2, False) + b.als_half_bytes(I, U, N, k, 2, False)
    assert abs(fp32 / 1e9 - 13.3) < 0.1  # "≈ 13.4 GB/epoch" with the OtOr pass
    assert abs(bf16 / 1e9 - 6.9) < 0.1  # "bf16 gather ≈ 7.0 GB"
    with_otor = b.als_half_bytes(U, I, N, k, 4, True) + b.als_half_bytes(I, U, N, k, 4, True)
    assert abs(with_otor / 1e9 - 13.4) < 0.1
    # 2.0 ms / 1.05 ms at the measured 6,571 GB/s
    assert abs(fp32 / 6571.2e9 * 1e3 - 2.03) < 0.05 and abs(bf16 / 6571.2e9 * 1e3 - 1.05) < 0.05


def test_knn_algorithmic_bytes_match_survey():
    b = _bench()
    # P = 1.278e10 products => 102 GB streamed, 15.6 ms at peak (SURVEY.md §8d)
    by = b.knn_build_bytes(12_764_118_364, 25_000_095, 162_541, 59_047, 1_180_940)
    assert abs(by / 1e9 - 102.3) < 0.5
    assert abs(by / 6571.2e9 * 1e3 - 15.6) < 0.2


def test_host_threads_ignores_omp_env(monkeypatch):
    b = _bench()
    monkeypatch.setenv("OMP_NUM_THREADS", "1")  # what torchrun exports to every rank
    import os

    assert b.host_threads() == len(os.sched_getaffinity(0)) >= 1


def test_committed_bench_lines_have_the_contract_keys():
    """The bench lines kept under profiles/ carry every key the driver's contract names."""
    need = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"}  # fmt: skip
    for name in ("r01_final_bench_n1.json", "r01_final_bench_n2.json", "r01_final_bench_n4.json"):
        line = json.loads((ROOT / "profiles" / name).read_text().strip().splitlines()[-1])
        assert need <= set(line), (name, need - set(line))
        assert line["vs_baseline"] is None and line["higher_is_better"] is False
        assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(line["roofline"])
        assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])
        assert "workload" in line["config"]
    ref = json.loads((ROOT / "profiles" / "r01_final_bench_reference_arm.json").read_text().strip().splitlines()[-1])
    assert ref["impl"] == "reference" and ref["e2e"]["h2d_bytes_per_step"] == 0
    assert {"kind", "cores", "sample", "value"} <= set(ref["cpu_baseline"])


def test_solve_cholesky_property():
    """The reference's property test of `solve_cholesky` (tests/utils/test_math_solve.py:21-50) against the
    host fold-in solver that mirrors it (`lkpy_b200.als._solve_cholesky`)."""
    import numpy as np
    from pytest import approx

    from lkpy_b200.als import _solve_cholesky

    for seed in range(40):
        rng = np.random.RandomState(seed)
        size = int(rng.randint(2, 101))
        A = rng.randn(size, size) * 10
        b = rng.randn(size) * 10
        A = A * A
        xexp = np.linalg.lstsq(A, b, rcond=None)[0]
        F, y = A.T @ A, A.T @ b
        x = _solve_cholesky(F, y)
        assert x.shape == y.shape
        assert x == approx(xexp, rel=1.0e-3)
        assert F @ x == approx(y, rel=2.0e-6, abs=5.0e-9)


def test_accel_mirror_signatures_match_reference_stubs():
    """Every function the reference's typed stubs declare for the two hot paths (`_accel/als.pyi`,
    `_accel/knn.pyi`; their parameter lists are recorded in tests/golden/reference_classes.npz) exists in
    lkpy_b200.accel with the same parameter names in the same order — the call sites (als/_implicit.py:161-164,
    als/_explicit.py:115-118, knn/item.py:162-171, :273-287, knn/user.py:224-240) bind positionally."""
    import inspect

    from lkpy_b200 import accel

    with np.load(ROOT / "tests" / "golden" / "reference_classes.npz") as z:
        stubs = {k: list(z[k]) for k in z.files if k.startswith("stubs/")}
    for mod, ns in (("als", accel.als), ("knn", accel.knn)):
        fns = stubs[f"stubs/{mod}"]
        assert fns
        for fn in fns:
            ours = getattr(ns, fn, None)
            assert ours is not None, f"_accel.{mod}.{fn} missing from the mirror"
            want = stubs[f"stubs/{mod}.{fn}"]
            got = list(inspect.signature(ours).parameters)
            assert got == want, (fn, got, want)
    # user-kNN scoring lives in the Rust module without a stub entry: same argument order as user_score.rs:21-29
    got = list(inspect.signature(accel.knn.user_score_items_explicit).parameters)
    assert got == ["tgt_items", "nbr_rows", "nbr_sims", "ratings", "max_nbrs", "min_nbrs"]


def test_accel_task_protocol_without_device():
    """invoke-once, cancel-before-invoke and progress shape of the task mirror (tasks/mod.rs:62-106) — host only."""
    from lkpy_b200.accel import AccelTask, run_accel_task

    t = AccelTask(lambda task: 7, total=10)
    assert t.current_progress() == (0, 10)
    assert run_accel_task(t) == 7
    assert t.current_progress() == (10, 10)
    with pytest.raises(RuntimeError, match="already invoked"):
        t.invoke()
    t2 = AccelTask(lambda task: 1, total=None)
    assert t2.current_progress() is None
    t2.cancel()
    with pytest.raises(RuntimeError, match="cancelled"):
        t2.invoke()
    with pytest.raises(RuntimeError, match="accelerator task failed"):
        run_accel_task(AccelTask(lambda task: 1 / 0))


def test_arrow_csr_ingest_and_chunks():
    """Arrow List / LargeList<Struct{index,value}> -> host CSR views -> LargeList chunks (csr.rs:160-209,
    consumer.rs:96-142) round-trip without a device."""
    import pyarrow as pa

    from lkpy_b200 import accel
    from lkpy_b200.data import InteractionCSR

    rng = np.random.default_rng(1)
    lens = rng.integers(0, 7, 50)
    indptr = np.concatenate([[0], np.cumsum(lens)])
    cols = np.concatenate([np.sort(rng.choice(40, n, replace=False)) for n in lens]).astype(np.int32)
    vals = rng.standard_normal(len(cols)).astype(np.float32)
    csr = InteractionCSR(indptr.astype(np.int64), cols, vals, (50, 40))
    chunks = accel.csr_to_arrow_chunks(csr, 16)
    assert len(chunks) == 4 and all(pa.types.is_large_list(c.type) for c in chunks)
    back = accel.as_host_csr(pa.chunked_array(chunks), 40)
    assert np.array_equal(back.indptr, csr.indptr) and np.array_equal(back.indices, cols)
    assert np.array_equal(back.values.view(np.int32), vals.view(np.int32)) and back.shape == (50, 40)
    # a sliced List array (non-zero first offset) and a structure-only array
    small = pa.ListArray.from_arrays(
        pa.array(indptr.astype(np.int32)),
        pa.StructArray.from_arrays([pa.array(cols), pa.array(vals)], names=["index", "value"]),
    ).slice(10, 20)
    sl = accel.as_host_csr(small, 40)
    assert sl.shape == (20, 40) and sl.indptr[0] == 0 and sl.nnz == int(indptr[30] - indptr[10])
    assert np.array_equal(sl.indices, cols[indptr[10] : indptr[30]])
    only = accel.as_host_csr(pa.ListArray.from_arrays(pa.array(indptr.astype(np.int32)), pa.array(cols)), 40)
    assert np.all(only.values == 1.0) and np.array_equal(only.indices, cols)


def test_row_part_length_by_kernel_path():
    """ALSTrainerBase._chunk_nnz: which row-part length each kernel path is planned with (DESIGN.md §4.2-4.3: the
    tensor-core accumulators add with round-toward-zero, so the tf32 paths and k = 128 get shorter parts)."""
    from types import SimpleNamespace

    from lkpy_b200 import _lib, engine
    from lkpy_b200.als import ALSTrainerBase

    def chunk(k, gather, mode=_lib.LK_ALS_IMPLICIT, use_ratings=False):
        me = SimpleNamespace(MODE=mode, config=SimpleNamespace(gather_dtype=gather, use_ratings=use_ratings))
        return ALSTrainerBase._chunk_nnz(me, k)

    assert chunk(64, "bfloat16") == engine.DEFAULT_CHUNK_NNZ  # als_tc_kernel: one accumulation per 16 rows
    assert chunk(64, "float32") == engine.TF32_CHUNK_NNZ  # als_tcx_kernel
    assert chunk(64, "bfloat16", use_ratings=True) == engine.TF32_CHUNK_NNZ  # weighted: tf32 path as well
    assert chunk(64, "float32", mode=_lib.LK_ALS_EXPLICIT) == engine.TF32_CHUNK_NNZ
    assert chunk(128, "bfloat16") == engine.TF32_CHUNK_NNZ  # als_tc128_kernel, kind::f16
    assert chunk(128, "float32") == engine.TF32_CHUNK_NNZ_K128  # als_tc128_kernel, tf32 x3
    assert chunk(128, "bfloat16", use_ratings=True) == engine.TF32_CHUNK_NNZ_K128
    assert chunk(32, "float32") == engine.DEFAULT_CHUNK_NNZ  # SIMT kernel
    assert engine.TF32_CHUNK_NNZ_K128 < engine.TF32_CHUNK_NNZ < engine.DEFAULT_CHUNK_NNZ


def test_synthetic_matrix_cache_round_trip(tmp_path):
    """data.synth_interactions_cached: the cached arrays are the generator's own, and a cache of another shape is
    not reused."""
    from lkpy_b200 import data

    shape = dict(n_users=400, n_items=150, nnz=6000)
    f = str(tmp_path / "cache.npz")
    a = data.synth_interactions_cached(f, **shape)
    b = data.synth_interactions_cached(f, **shape)  # from the file
    c = data.synth_interactions(**shape)
    for x in (a, b):
        assert (x.n_users, x.n_items) == (c.n_users, c.n_items)
        assert np.array_equal(x.users, c.users) and np.array_equal(x.items, c.items)
        assert np.array_equal(x.ratings.view(np.int32), c.ratings.view(np.int32))
    other = data.synth_interactions_cached(f, n_users=300, n_items=150, nnz=5000)
    assert other.n_users == 300 and other.nnz == 5000
    assert data.synth_interactions_cached(None, **shape).nnz == c.nnz


def test_own_index_type_matches_the_reference_wire_format():
    """Without lenskit in the process the index field of a result carries this package's own class of the
    ``lenskit.sparse_index`` extension type: same name, same JSON metadata (data/matrix.py:104-146), unregistered."""
    import json
    import sys

    import pyarrow as pa

    from lkpy_b200 import accel

    if "lenskit.data.matrix" in sys.modules:
        pytest.skip("lenskit is loaded: its own class is used")
    t = accel.sparse_index_type(9066)
    assert t.extension_name == "lenskit.sparse_index" and t.storage_type == pa.int32() and t.dimension == 9066
    assert json.loads(t.__arrow_ext_serialize__().decode()) == {"dimension": 9066}
    assert type(t).__arrow_ext_deserialize__(pa.int32(), t.__arrow_ext_serialize__()).dimension == 9066
