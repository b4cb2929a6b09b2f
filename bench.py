#!/usr/bin/env python
"""
bench.py — ALS-implicit epoch time and item-kNN build / score throughput on
ML-25M-shaped synthetic interactions (BASELINE.json metric; configs[1], configs[2]) and the two
scale-out configurations (configs[3], configs[4]).

    python bench.py --gpus 1 --steps 20 --warmup 3                 # the default line (configs[1] + [2])
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...                            # CPU restatement of the reference path
    ... bench.py --gpus 8 --workload als100m                        # configs[3]: 100 M interactions, k=128
    ... bench.py --gpus 8 --workload knn1b                          # configs[4]: 1 B interactions, kNN build

One JSON line on stdout (rank 0).  A "step" is one ALS epoch (user half-epoch + item half-epoch,
each = OtOr kernel + row-solve kernel, + the factor exchange when N > 1) over the resident CSR
matrices.  `value` is the epoch time with everything resident in HBM; `e2e` is the same epoch
through the public trainer API with the factor tables coming from / going back to pinned host
memory inside the timed region.  Riding along in the same line:
  "als_fp32"   the same epoch with fp32 gathered rows (the like-for-like figure against the f32 reference),
  "knn"        item-kNN build items/s (kernel roofline, CPU baseline, e2e through the plugin call
               `accel.compute_similarities` with host CSR in / host CSR out, and through
               `ItemKNNScorer.train`), batched scoring of ALL users against all items (users/s, roofline),
  "recommend"  (N=1) batched ALS scoring + top-100 users/s,
  "parity"     oracle checks at THIS shape, run after the timed loops: sampled rows of one ALS
               half-step (bf16 and fp32 rows; split / empty / short rows included) against the f64 oracle,
               sampled item-kNN rows bit-exact against the oracle, and at N > 1 cross-rank equality of
               the replicas + equality with a single-GPU half-step.  A mismatch makes the run exit 1.
"cpu_baseline" and `--impl reference` time the CPU restatement of the reference path (oracle/) on a
bounded sample: median of 3 repeats, thread sweep including the reference's default of 8 threads.
Only the JSON line goes to stdout.

`--dump-outputs DIR` writes, after the timed loops, what each timed path computed in its last timed step as
DIR/<name>.npy (float32 / float64, integers stored exactly): the factor tables after the last timed ALS epoch
(a fixed, seeded sample of rows), the item-kNN similarity matrix of the last timed build (CSR), and a seeded
sample of query rows of the last scoring launch (scores with 0 where an item is unscored, a 0/1 mask of the
scored items, and neighbour counts).  Inputs are seeded, so two builds of the project run with the
same arguments can be compared output for output.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

METRIC = "als_implicit_epoch_time_ml25m_k64"
UNIT = "ms"
K = 64
WEIGHT = 40.0
REG = 0.1
KNN_SAVE = 20
KNN_MIN_SIM = 1e-6
KNN_MAX_NBRS = 20


def log(*a):
    if int(os.environ.get("RANK", "0")) == 0:
        print(*a, file=sys.stderr, flush=True)


# ---------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = (
        "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
        "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    )

    def __init__(self, gpu_index: int = 0):
        self.rows: list = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )  # fmt: skip
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        assert self.proc and self.proc.stdout
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def wait_first(self, timeout: float = 8.0) -> None:
        """nvidia-smi takes a few hundred ms to print its first row: block until it is sampling."""
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.02)

    def stop(self, t_begin: float | None = None, t_end: float | None = None) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        rows = list(self.rows)
        window = "timed region"
        if t_begin is not None and t_end is not None:
            inside = [r for t, r in rows if t_begin <= t <= t_end + 0.02]
            if len(inside) >= 2:
                sel = inside
            else:  # region shorter than two sampling periods: use the samples under the same load around it
                sel = [r for t, r in rows if t_begin - 0.5 <= t <= t_end + 0.1]
                window = "timed region +/- warm-up epochs (region shorter than two 20 ms samples)"
        else:
            sel = [r for _, r in rows]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in sel:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except (ValueError, IndexError):
                continue
        return {
            "sm_mhz": float(np.median(sm)) if sm else None,
            "sm_max_mhz": float(max(mx)) if mx else None,
            "samples": len(sm),
            "window": window,
            "reasons": sorted(reasons),
        }


# ---------------------------------------------------------------------------
# algorithmic bytes (SURVEY.md §8d, DESIGN.md §roofline)
# ---------------------------------------------------------------------------


def als_half_bytes(n_rows: int, n_other: int, nnz: int, k: int, s: int, with_otor: bool) -> float:
    b = nnz * (k * s + 8) + 4 * (n_rows + 1) + n_rows * k * 4 * 2 + k * k * 4
    if with_otor:
        b += n_other * k * 4 + (n_other * k * 2 if s == 2 else 0)
    return float(b)


def knn_build_bytes(products: int, nnz: int, n_users: int, n_items: int, nnz_out: int) -> float:
    return float(8 * products + 8 * nnz + 4 * (n_items + n_users + 2) + 8 * nnz_out)


def knn_score_bytes(sim_entries_touched: int, hist: int, targets: int) -> float:
    """SURVEY.md §8d: 8·Σ_{r∈hist}|S.row(r)| + 8·|hist| + 8·|targets| (summed over the batch)."""
    return float(8 * sim_entries_touched + 8 * hist + 8 * targets)


def load_peaks() -> tuple[float, str]:
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(key: str, world: int) -> float | None:
    """DRAM bytes per launch from the committed ncu --set full capture (N=1, default workload only)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        f = ROOT / "profiles" / name
        if world == 1 and f.exists():
            v = json.loads(f.read_text()).get(key)
            if v:
                return float(v)
    return None


# ---------------------------------------------------------------------------
# CPU baseline (oracle port of src/accel; the Rust crate cannot be built here)
# ---------------------------------------------------------------------------


def host_threads() -> int:
    """
    Host threads the CPU arm may use: the cores this process may run on.  (Not OMP_NUM_THREADS:
    torchrun exports OMP_NUM_THREADS=1 to every rank, which would silently turn the multi-threaded
    CPU baseline into a single-threaded one whenever the bench is launched under it.)
    """
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:  # pragma: no cover
        return max(1, os.cpu_count() or 1)


def thread_candidates(top: int) -> list[int]:
    """All host threads, half of them, and 8 = the reference's default pool (schemas/settings.py:182-185)."""
    return sorted({t for t in (top, max(top // 2, 1), 32, 8) if 1 <= t <= top}, reverse=True)


def _slice_rows(csr, lo: int, hi: int):
    from lkpy_b200.data import InteractionCSR

    a, b = int(csr.indptr[lo]), int(csr.indptr[hi])
    return InteractionCSR(
        (csr.indptr[lo : hi + 1] - a).astype(np.int64), csr.indices[a:b], csr.values[a:b], (hi - lo, csr.shape[1])
    )


def cpu_als_epoch_estimate(ui, iu, p, q, budget_s: float, threads: int, k: int = K) -> dict:
    """
    The ALS half-epochs of the reference path on the host (oracle/lk_cpu_fast.c: thread-private
    register-blocked Gram + vectorised Cholesky, scales with the cores) on leading row ranges of both
    halves (rows are in random order with respect to length: user weights and the item permutation
    are i.i.d.), scaled by nnz to a full epoch.  Per half: a calibration slice picks the sample
    size for the budget, then every thread count in `thread_candidates` is timed three times on the
    SAME sample and the median kept; the figure reported is the fastest thread count's median, the
    8-thread figure (the reference's default pool) rides along.
    """
    import oracle

    total_best, total_8 = 0.0, 0.0
    parts, per_threads = [], {}
    cands = thread_candidates(threads)
    best_threads = []
    for name, csr, this, other in (("user", ui, p, q), ("item", iu, q, p)):
        o32 = (other.T @ other + np.eye(k, dtype=np.float32) * REG).astype(np.float32)
        nnz = csr.nnz
        rows_cal = max(int(np.searchsorted(csr.indptr, nnz // 50)), 16)
        cal = _slice_rows(csr, 0, rows_cal)
        oracle.als_half_fast("implicit", cal, this[:rows_cal], other, otor_mat=o32, threads=cands[0])  # pool start-up
        t0 = time.perf_counter()
        oracle.als_half_fast("implicit", cal, this[:rows_cal], other, otor_mat=o32, threads=cands[0])
        t_cal = time.perf_counter() - t0
        nnz_cal = int(csr.indptr[rows_cal])
        per_run = budget_s / 2 / (3 * len(cands))  # three repeats per thread count, two halves
        want_nnz = int(min(nnz, nnz_cal * per_run / max(t_cal, 1e-6)))
        rows = int(np.searchsorted(csr.indptr, want_nnz))
        rows = min(max(rows, rows_cal), csr.shape[0])
        sample = _slice_rows(csr, 0, rows)
        nnz_s = int(csr.indptr[rows])
        med = {}
        for th in cands:
            ts = []
            for _rep in range(3):
                t0 = time.perf_counter()
                oracle.als_half_fast("implicit", sample, this[:rows], other, otor_mat=o32, threads=th)
                ts.append(time.perf_counter() - t0)
            med[th] = float(np.median(ts)) * nnz / max(nnz_s, 1)
        bt = min(med, key=med.get)
        best_threads.append(bt)
        total_best += med[bt]
        total_8 += med.get(8, med[min(med)])
        for th, v in med.items():
            per_threads[th] = per_threads.get(th, 0.0) + v * 1e3
        parts.append(f"{name} half: rows 0..{rows} ({nnz_s} nnz = {nnz_s / nnz:.1%}), best at {bt} threads")
    return {
        "epoch_ms": total_best * 1e3,
        "epoch_ms_8_threads": total_8 * 1e3,
        "threads": max(best_threads),
        "epoch_ms_by_threads": {str(t): round(v, 2) for t, v in sorted(per_threads.items())},
        "sample": "; ".join(parts) + "; median of 3 per thread count, scaled by nnz to the full epoch",
    }


def cpu_knn_estimate(kui, kiu, cost: np.ndarray, budget_s: float, threads: int) -> dict:
    """
    Item-kNN build of the reference path on the host (oracle sim_row, thread-private accumulators)
    on a FIXED stratified sample: items sorted by product count, every `stride`-th one taken, so the
    sample carries the cost distribution of the whole matrix (hot items included in proportion);
    median of 3 per thread count; scaled by product count.
    """
    import oracle

    n_items = kiu.shape[0]
    total_cost = float(cost.sum())
    order = np.argsort(-cost, kind="stable")
    cands = thread_candidates(threads)
    # calibrate on a 1/200 systematic sample
    cal = order[100::200]
    oracle.knn_build(kui, kiu, KNN_MIN_SIM, KNN_SAVE, row_list=cal, threads=cands[0])
    t0 = time.perf_counter()
    oracle.knn_build(kui, kiu, KNN_MIN_SIM, KNN_SAVE, row_list=cal, threads=cands[0])
    t_cal = time.perf_counter() - t0
    per_run = budget_s / (3 * len(cands))
    frac = min(1.0, (float(cost[cal].sum()) / total_cost) * per_run / max(t_cal, 1e-6))
    stride = max(1, int(round(1.0 / max(frac, 1e-9))))
    sample = order[stride // 2 :: stride]
    c = float(cost[sample].sum())
    med = {}
    for th in cands:
        ts = []
        for _rep in range(3):
            t0 = time.perf_counter()
            oracle.knn_build(kui, kiu, KNN_MIN_SIM, KNN_SAVE, row_list=sample, threads=th)
            ts.append(time.perf_counter() - t0)
        med[th] = float(np.median(ts)) * total_cost / max(c, 1.0)
    bt = min(med, key=med.get)
    return {
        "build_items_per_s": n_items / med[bt],
        "threads": bt,
        "items_per_s_by_threads": {str(t): round(n_items / v, 1) for t, v in sorted(med.items())},
        "sample": (f"every {stride}-th item of the cost-sorted list ({len(sample)} items, {c / total_cost:.2%} of the "
                   f"products), median of 3 per thread count, scaled by product count"),
    }  # fmt: skip


# ---------------------------------------------------------------------------
# data
# ---------------------------------------------------------------------------


def make_data():
    from lkpy_b200 import data

    t0 = time.time()
    inter = data.synth_interactions_cached(os.environ.get("LK_BENCH_DATA_CACHE"), **data.ML25M_SHAPE)
    log(f"[bench] synthetic ML-25M-shaped data: {inter.n_users}x{inter.n_items}, nnz {inter.nnz} ({time.time() - t0:.1f}s)")
    return inter


def run_reference(args, rank: int) -> None:
    """--impl reference: the CPU path (oracle port; Rust unavailable) on a bounded sample."""
    if rank != 0:
        return
    from lkpy_b200 import data

    inter = make_data()
    ui, iu = data.als_implicit_matrices(inter, WEIGHT)
    rng = np.random.default_rng(0)
    p = (rng.standard_normal((inter.n_users, K)) * 0.1).astype(np.float32)
    q = (rng.standard_normal((inter.n_items, K)) * 0.1).astype(np.float32)
    threads = host_threads()
    per_step = max(6.0, 150.0 / max(args.steps + args.warmup, 1))
    vals, sample, r = [], "", {}
    for s in range(args.warmup + args.steps):
        r = cpu_als_epoch_estimate(ui, iu, p, q, per_step, threads)
        if s >= args.warmup:
            vals.append(r["epoch_ms"])
        sample = r["sample"]
    v = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": v, "higher_is_better": False,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "ML-25M-shaped synthetic ImplicitMFScorer features=64 (configs[1])",
                   "n_users": inter.n_users, "n_items": inter.n_items, "nnz": inter.nnz},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": r.get("threads"), "kind": "port", "sample": sample,
                         "epoch_ms_by_threads": r.get("epoch_ms_by_threads"),
                         "epoch_ms_8_threads": r.get("epoch_ms_8_threads")},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }  # fmt: skip
    emit(line)


_JSON_OUT = None


DUMP_LIMIT = 64 << 20  # bytes written by --dump-outputs in all
DUMP_ROWS = 16384  # sampled rows per factor table


def sample_rows(n: int, k: int, seed: int) -> np.ndarray:
    """A fixed, sorted sample of ``min(n, k)`` row indices."""
    return np.sort(np.random.default_rng(seed).choice(n, min(n, k), replace=False))


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """``--dump-outputs``: one ``<name>.npy`` per array, finite float32 / float64 only, within DUMP_LIMIT."""
    total = sum(np.asarray(a).nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        assert np.isfinite(a).all(), f"--dump-outputs: {name} is not finite"
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    log(f"[bench] wrote {len(arrays)} arrays ({total} bytes) to {out_dir}")


def emit(line: dict) -> None:
    """The one JSON line goes to the real stdout; everything else (NCCL's version banner, library
    chatter written to fd 1) was redirected to stderr by main()."""
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


# ---------------------------------------------------------------------------
# parity at the benchmark's own shape (after the timed loops)
# ---------------------------------------------------------------------------


def als_parity(tr, inter, tag: str, rank: int, world: int, dev) -> dict | None:
    """
    One user half-step and one item half-step from fixed trained-scale factors on the trainer that was
    just timed (single-GPU or sharded); rank 0 compares sampled rows with the f64 oracle
    (oracle/parity.py).  At N > 1 additionally: the replicas of all ranks carry the same bits, and they
    equal a single-GPU half-step run on rank 0.
    """
    import torch

    from lkpy_b200 import engine

    bf16 = tag == "bf16"
    rng = np.random.default_rng(1234)
    p0 = (rng.standard_normal((inter.n_users, K)) * 0.1).astype(np.float32)
    q0 = (rng.standard_normal((inter.n_items, K)) * 0.1).astype(np.float32)
    tp0, tq0 = torch.from_numpy(p0).to(dev), torch.from_numpy(q0).to(dev)
    sharded = world > 1

    def half(which: str):
        tr.d_users.copy_(tp0)
        tr.d_items.copy_(tq0)
        tr.u_plan.status.zero_()
        tr.i_plan.status.zero_()
        if sharded:
            import torch.distributed as dist

            torch.cuda.synchronize()
            dist.barrier()  # every replica holds (P0, Q0) before anyone's kernel writes into it
            tr.half_step(which)
            torch.cuda.synchronize()
            dist.barrier()
        elif which == "user":
            tr._half(tr.u_plan, tr.d_users, tr.d_items, tr.d_items_bf16, tr.config.user_reg)
        else:
            tr._half(tr.i_plan, tr.d_items, tr.d_users, tr.d_users_bf16, tr.config.item_reg)
        torch.cuda.synchronize()
        tr._raise_on_status()
        return (tr.d_users if which == "user" else tr.d_items).clone()

    new_p = half("user")
    new_q = half("item")
    out: dict = {}
    if sharded:
        import torch.distributed as dist

        from oracle import parity

        cs = parity.checksum(new_p.cpu().numpy(), new_q.cpu().numpy())
        # 64-bit checksums compared as two 32-bit halves (NCCL has no u64 min/max on every build)
        t = torch.tensor([cs >> 32, cs & 0xFFFFFFFF], dtype=torch.int64, device=dev)
        lo, hi = t.clone(), t.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        out["replicas_equal_across_ranks"] = bool(torch.equal(lo, hi))
    if rank != 0:
        return None
    from oracle import parity

    ui, iu = tr.ui_host, tr.iu_host
    res = {}
    for which, csr, old, other, new in (("user", ui, p0, q0, new_p), ("item", iu, q0, p0, new_q)):
        rows = parity.sample_als_rows(csr.indptr, K, engine.DEFAULT_CHUNK_NNZ, seed=7)
        got = new[torch.from_numpy(rows).to(dev)].cpu().numpy()
        res[which] = parity.check_als_half("implicit", csr, rows, old[rows], other, got, REG, bf16)
    out.update(res)
    out["ok"] = bool(res["user"]["ok"] and res["item"]["ok"] and out.get("replicas_equal_across_ranks", True))
    if sharded:
        # the same two half-steps on one GPU (rank 0, full matrices): sharding must not change a bit
        from lkpy_b200.als import ImplicitMFScorer, ImplicitMFTrainer
        from lkpy_b200.components import Dataset, TrainingOptions

        sc = ImplicitMFScorer(features=K, epochs=1, regularization=REG, weight=WEIGHT, gather_dtype=tr.config.gather_dtype)
        single = ImplicitMFTrainer(sc, Dataset(inter), TrainingOptions(rng=42))
        single.d_users.copy_(tp0)
        single.d_items.copy_(tq0)
        single._half(single.u_plan, single.d_users, single.d_items, single.d_items_bf16, REG)
        eq_u = bool(torch.equal(single.d_users, new_p))
        single.d_users.copy_(tp0)
        single._half(single.i_plan, single.d_items, single.d_users, single.d_users_bf16, REG)
        eq_i = bool(torch.equal(single.d_items, new_q))
        out["equals_single_gpu_half_step"] = {"user": eq_u, "item": eq_i}
        out["ok"] = bool(out["ok"] and eq_u and eq_i)
        del single
        torch.cuda.empty_cache()
    log(f"[bench] parity ALS {tag}: user {res['user']['rel_fro_vs_f64_oracle']:.2e} "
        f"item {res['item']['rel_fro_vs_f64_oracle']:.2e} (tol 1e-4) "
        + (f"unrounded-oracle distance {res['user'].get('rel_fro_vs_unrounded_f64_oracle', 0):.2e} / "
           f"{res['item'].get('rel_fro_vs_unrounded_f64_oracle', 0):.2e} " if bf16 else "")
        + f"ok={out['ok']}")  # fmt: skip
    return out


# ---------------------------------------------------------------------------
# main
# ---------------------------------------------------------------------------


def main() -> None:
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ml25m", choices=["ml25m", "als100m", "knn1b"])
    ap.add_argument("--cpu-seconds", type=float, default=18.0, help="CPU baseline budget per path")
    ap.add_argument("--no-knn", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--score-batch", type=int, default=16384,
                    help="users per scoring launch (all users are scored); a launch lasts at least as long as its "
                         "heaviest query (2.6 ms at ML-25M shape), so small batches are tail-bound")
    ap.add_argument("--score-users", type=int, default=0, help="score only this many users (0 = all)")
    ap.add_argument("--variants", default="bf16,fp32", help="ALS gather dtypes to time (profiling runs pass one)")
    ap.add_argument("--profile", action="store_true", help="under ncu: honour a small --warmup, skip e2e/parity/CPU")
    ap.add_argument("--scale", type=float, default=1.0, help="scale-out workloads: fraction of the full size (smoke runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed paths computed in their last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)
    if args.profile:
        args.no_parity = args.no_cpu = True

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch

    from lkpy_b200 import _build, _lib, data
    from lkpy_b200.als import ImplicitMFScorer, ImplicitMFTrainer
    from lkpy_b200.components import Dataset, TrainingOptions

    _build.build()
    _lib.lib()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    peak, peak_src = load_peaks()

    if args.workload != "ml25m":
        import bench_scale

        line = bench_scale.run(args, rank, world, dev, peak, peak_src)
        if rank == 0:
            emit(line)
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()
        return

    inter = make_data()
    ds = Dataset(inter)

    def barrier():
        if world > 1:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    results: dict = {}
    parity: dict = {}
    dumped: dict = {}  # --dump-outputs, rank 0
    launches = 0
    variants = [v for v in args.variants.split(",") if v]
    for tag, gdt in (("bf16", "bfloat16"), ("fp32", "float32")):
        if tag not in variants:
            continue
        scorer = ImplicitMFScorer(features=K, epochs=1, regularization=REG, weight=WEIGHT, gather_dtype=gdt)
        if world > 1:
            from lkpy_b200.parallel import ShardedImplicitMFTrainer

            tr = ShardedImplicitMFTrainer(scorer, ds, TrainingOptions(rng=42))
        else:
            tr = ImplicitMFTrainer(scorer, ds, TrainingOptions(rng=42))
        # one epoch from the reference init first, so timed epochs see trained-scale factors
        for _ in range(args.warmup if args.profile else max(args.warmup, 3)):
            tr.train_epoch_device()
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0 and tag == "bf16":
            sampler.start()
            sampler.wait_first()
        if tag == "bf16":
            for _ in range(3):  # every rank: the GPU stays under the same load while the sampler spins up
                tr.train_epoch_device()
        graphed = bool(world > 1 and not args.profile and tr.enable_graph())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t_begin = time.time()
        e0.record()
        for _ in range(args.steps):
            tr.train_epoch_device()
        e1.record()
        barrier()
        t_end = time.time()
        clocks = sampler.stop(t_begin, t_end) if (rank == 0 and tag == "bf16") else None
        if args.dump_outputs and rank == 0:  # the factors as the last timed epoch left them
            for side, t, seed in (("user", tr.d_users, 1), ("item", tr.d_items, 2)):
                rows = torch.from_numpy(sample_rows(t.shape[0], DUMP_ROWS, seed)).to(t.device)
                dumped[f"als_{tag}_{side}_rows"] = rows.cpu().numpy().astype(np.float64)
                dumped[f"als_{tag}_{side}_factors"] = t.index_select(0, rows).float().cpu().numpy()
        # the same epochs once more with CUDA events around every row-solve launch (the roofline's
        # kernel time; events cannot sit inside a captured graph, so this loop launches eagerly)
        tr.kernel_events = []
        for _ in range(args.steps):
            tr.train_epoch_device()
        barrier()
        ms = e0.elapsed_time(e1) / args.steps
        kern_ms = [a.elapsed_time(b) for a, b in tr.kernel_events]
        tr.kernel_events = None
        tr._raise_on_status()
        if world > 1:
            import torch.distributed as dist

            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        s = 2 if tag == "bf16" else 4
        nnz = inter.nnz
        # per GPU: each rank gathers for its row shard only (1/world of the nonzeros and rows)
        alg = (
            als_half_bytes(inter.n_users, inter.n_items, nnz, K, s, False)
            + als_half_bytes(inter.n_items, inter.n_users, nnz, K, s, False)
        ) / world
        per_epoch_kernel_ms = float(np.sum(kern_ms)) / args.steps if kern_ms else float("nan")
        achieved = alg / (per_epoch_kernel_ms * 1e-3) / 1e9 if kern_ms else float("nan")
        results[tag] = {
            "ms_per_epoch": ms,
            "solve_kernel_ms_per_epoch": per_epoch_kernel_ms,
            "roofline": {
                "bound": "hbm",
                "kernel": tr.solve_kernel_name() + " (user + item launch of one epoch)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic("als_tc_kernel_epoch_bytes", world) if tag == "bf16" else None,
                "algorithmic_bytes": alg, "peak_source": peak_src,
            },
            "clocks": clocks,
            "cuda_graph": graphed,
        }  # fmt: skip
        launches = tr.launches_per_epoch() * args.steps
        log(f"[bench] ALS {tag}: {ms:.3f} ms/epoch (solve kernels {per_epoch_kernel_ms:.3f} ms), "
            f"{achieved:.0f} GB/s algorithmic = {achieved / peak:.3f} of {peak_src}")

        # ---- end to end through the trainer API: factors from / to pinned host memory
        if not args.profile:
            if world > 1:
                # ONE host model shared by the ranks (/dev/shm, page-locked in every process)
                from lkpy_b200.parallel import shared_pinned_tensor

                names = (f"lkpy_b200_bench_p_{os.environ.get('MASTER_PORT', '0')}",
                         f"lkpy_b200_bench_q_{os.environ.get('MASTER_PORT', '0')}")
                shapes = (tuple(tr.d_users.shape), tuple(tr.d_items.shape))
                if rank == 0:
                    hp, hq = (shared_pinned_tensor(n, sh, create=True) for n, sh in zip(names, shapes))
                    hp.copy_(tr.d_users)
                    hq.copy_(tr.d_items)
                barrier()
                if rank != 0:
                    hp, hq = (shared_pinned_tensor(n, sh) for n, sh in zip(names, shapes))
                barrier()
                if rank == 0:
                    for n in names:
                        os.unlink(f"/dev/shm/{n}")  # the mappings stay valid
            else:
                hp = torch.from_numpy(scorer.user_embeddings).pin_memory()
                hq = torch.from_numpy(scorer.item_embeddings).pin_memory()
            for _ in range(2):
                tr.train_epoch_e2e(hp, hq)
            barrier()
            t0 = time.perf_counter()
            e0.record()
            for _ in range(args.steps):
                tr.train_epoch_e2e(hp, hq)
            e1.record()
            barrier()
            wall = (time.perf_counter() - t0) * 1e3 / args.steps
            e2e_ms = e0.elapsed_time(e1) / args.steps
            nbytes = (hp.numel() + hq.numel()) * 4
            h2d, d2h = nbytes, nbytes + 16
            api = "ImplicitMFTrainer.train_epoch_e2e: H2D factor tables, epoch, D2H factor tables + deltas; CSR resident"
            if world > 1:
                import torch.distributed as dist

                # every rank moves the rows it owns (the PCIe links work in parallel): sum over ranks
                t = torch.tensor([tr.e2e_bytes[0], tr.e2e_bytes[1], max(e2e_ms, wall)], device=dev, dtype=torch.float64)
                tmax = t.clone()
                dist.all_reduce(t)
                dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
                h2d, d2h = int(t[0].item()), int(t[1].item())
                e2e_ms = wall = float(tmax[2].item())
                api = ("ShardedImplicitMFTrainer.train_epoch_e2e: each rank uploads and downloads the row shards it "
                       "owns into one shared pinned host model; bytes summed over ranks")
            results[tag]["e2e"] = {
                "value": max(e2e_ms, wall), "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "api": api,
            }  # fmt: skip
            log(f"[bench] ALS {tag} e2e: {results[tag]['e2e']['value']:.3f} ms/epoch")
            if world > 1:
                from lkpy_b200.parallel import release_shared_pinned

                barrier()
                release_shared_pinned(hp)
                release_shared_pinned(hq)
            del hp, hq
            if tag == "bf16" and rank == 0 and world == 1 and not args.no_knn:
                results["recommend"] = bench_recommend(args, tr, dev, peak, peak_src)
        if not args.no_parity:
            r = als_parity(tr, inter, tag, rank, world, dev)
            if r is not None:
                parity["als_" + tag] = r
        del tr, scorer
        torch.cuda.empty_cache()

    knn = None
    if not args.no_knn:
        knn = bench_knn(args, inter, dev, peak, peak_src, rank, world, parity, dumped if args.dump_outputs else None)

    cpu = None
    if not args.no_cpu and rank == 0 and world == 1:
        threads = host_threads()
        ui, iu = data.als_implicit_matrices(inter, WEIGHT)
        rng = np.random.default_rng(0)
        p = (rng.standard_normal((inter.n_users, K)) * 0.1).astype(np.float32)
        q = (rng.standard_normal((inter.n_items, K)) * 0.1).astype(np.float32)
        r = cpu_als_epoch_estimate(ui, iu, p, q, args.cpu_seconds, threads)
        cpu = {"value": r["epoch_ms"], "unit": UNIT, "cores": r["threads"], "kind": "port", "sample": r["sample"],
               "epoch_ms_by_threads": r["epoch_ms_by_threads"], "epoch_ms_8_threads": r["epoch_ms_8_threads"],
               "host_threads": threads}  # fmt: skip
        log(f"[bench] CPU baseline ({r['threads']} threads): {r['epoch_ms']:.0f} ms/epoch "
            f"(by threads {r['epoch_ms_by_threads']})  [{r['sample']}]")
        if knn is not None and "_kui" in knn:
            kc = cpu_knn_estimate(knn["_kui"], knn["_kiu"], knn["_cost"], args.cpu_seconds, threads)
            knn["cpu_baseline"] = {"value": kc["build_items_per_s"], "unit": "items/s", "cores": kc["threads"],
                                   "kind": "port", "sample": kc["sample"],
                                   "items_per_s_by_threads": kc["items_per_s_by_threads"]}  # fmt: skip
            log(f"[bench] CPU kNN build: {kc['build_items_per_s']:.0f} items/s at {kc['threads']} threads "
                f"(by threads {kc['items_per_s_by_threads']}) [{kc['sample']}]")
    if knn is not None:
        for k_ in ("_kui", "_kiu", "_cost"):
            knn.pop(k_, None)

    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dumped)
    ok = all(v.get("ok", True) for v in parity.values()) if parity else None
    if rank == 0:
        head = results.get("bf16") or results["fp32"]
        parity["ok"] = ok
        line = {
            "metric": METRIC, "value": head["ms_per_epoch"], "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_epoch"],
            "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32 (bf16-stored gather operand)", "data": "synthetic",
            "config": {
                "workload": "ML-25M-shaped synthetic ImplicitMFScorer features=64 bf16 gather (BASELINE configs[1])",
                "n_users": inter.n_users, "n_items": inter.n_items, "nnz": inter.nnz, "features": K,
                "weight": WEIGHT, "reg": REG, "parallelism": f"row-sharded x{world}" if world > 1 else "single GPU",
                "l2": "inputs (2 CSR orientations 400 MB + factors) exceed the 126 MB L2; no explicit flush",
            },
            "roofline": head["roofline"], "clocks": head["clocks"], "e2e": head.get("e2e"),
            "cuda_graph": head.get("cuda_graph"),
            "gpu_launches": launches, "cpu_baseline": cpu,
            "als_fp32": ({"ms_per_epoch": results["fp32"]["ms_per_epoch"], "roofline": results["fp32"]["roofline"],
                          "e2e": results["fp32"].get("e2e")} if "fp32" in results else None),
            "knn": knn,
            "recommend": results.get("recommend"),
            "parity": parity if not args.no_parity else None,
        }  # fmt: skip
        emit(line)
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    if ok is False:
        log("[bench] PARITY FAILURE — see the `parity` object")
        raise SystemExit(1)


def dump_csr(dumped: dict, name: str, indptr, cols, vals) -> None:
    dumped[f"{name}_indptr"] = indptr.cpu().numpy().astype(np.float64)
    dumped[f"{name}_cols"] = cols.cpu().numpy().astype(np.float64)
    dumped[f"{name}_vals"] = vals.cpu().numpy().astype(np.float32)


def bench_recommend(args, tr, dev, peak, peak_src) -> dict:
    """
    SURVEY.md §8f N1/N2: top-100 of all items for a batch of users from the factors just trained —
    one fp32 library GEMM (Q · Xᵀ, item-major) + lk_topn_columns (the reference's heap, one thread
    per user).  CPU figure: the reference's per-query path (f32 matvec + argtopn), one thread.
    """
    import torch

    from lkpy_b200 import engine

    n_top, batch = 100, min(131072, int(tr.d_users.shape[0]))  # one thread per user: large batches fill the GPU
    q, p = tr.d_items, tr.d_users
    rng = np.random.default_rng(11)
    users = torch.from_numpy(np.sort(rng.choice(p.shape[0], batch, replace=False))).to(dev)
    x = p[users].contiguous()
    s = q @ x.T
    engine.topn_columns(s, n_top)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    reps = args.steps
    t_gemm = t_top = 0.0
    for _ in range(reps):
        ev[0].record()
        s = q @ x.T
        ev[1].record()
        idx, val, cnt = engine.topn_columns(s, n_top)
        ev[2].record()
        torch.cuda.synchronize()
        t_gemm += ev[0].elapsed_time(ev[1]) / reps
        t_top += ev[1].elapsed_time(ev[2]) / reps
    n_items = q.shape[0]
    alg = float(n_items) * batch * 4  # the selection reads every score once
    achieved = alg / (t_top * 1e-3) / 1e9
    out = {
        "workload": f"top-{n_top} of {n_items} items for {batch} trained users (ML-25M-shaped ImplicitMF k={K})",
        "users_per_s": batch / ((t_gemm + t_top) * 1e-3), "gemm_ms": t_gemm, "topn_ms": t_top,
        "roofline": {"bound": "hbm", "kernel": "topn_columns_kernel", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "traffic": None, "algorithmic_bytes": alg,
                     "peak_source": peak_src},
    }  # fmt: skip
    log(f"[bench] recommend: {batch} users x top-{n_top}: GEMM {t_gemm:.1f} ms + top-N {t_top:.1f} ms = "
        f"{out['users_per_s']:.0f} users/s; top-N {achieved:.0f} GB/s = {achieved / peak:.3f} of peak")
    if not args.no_cpu:
        import oracle

        qh, ph = q.cpu().numpy(), x[:256].cpu().numpy()
        t0 = time.perf_counter()
        done = 0
        for u in range(len(ph)):
            sc = qh @ ph[u]
            oracle.argtopn(sc, n_top)
            done += 1
            if time.perf_counter() - t0 > 4.0:
                break
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": done / dt, "unit": "users/s", "cores": 1, "kind": "port",
                               "sample": f"{done} users, f32 matvec + heap argtopn each, one thread"}  # fmt: skip
        # selection parity on the way: the device lists of the first users against the oracle on the device scores
        sh = s[:, :8].cpu().numpy()
        ih = idx[:8].cpu().numpy()
        for c in range(8):
            assert np.array_equal(ih[c], oracle.argtopn(sh[:, c], n_top)), "top-N mismatch vs oracle"
        log(f"[bench] CPU recommend: {out['cpu_baseline']['value']:.0f} users/s (one thread)")
    del s
    return out


def bench_knn(args, inter, dev, peak, peak_src, rank: int, world: int, parity: dict, dumped: dict | None = None) -> dict | None:
    import torch

    from lkpy_b200 import accel, data, engine
    from lkpy_b200.components import Dataset

    t0 = time.time()
    kui, kiu, means = data.knn_item_matrices(inter, True)
    prep_s = time.time() - t0
    log(f"[bench] kNN host prep {prep_s:.1f}s")
    d_ui = engine.DeviceCSR.from_host(kui, dev)
    d_iu = engine.DeviceCSR.from_host(kiu, dev)

    plan = engine.KnnBuildPlan.create(d_ui, d_iu, world=world)  # allocates the workspaces once
    cost = plan.cost.cpu().numpy()
    products = int(cost.sum()) - inter.nnz  # sim_row skips the diagonal entry of every (item, user) visit

    def score_users(st, R, u_begin: int, u_end: int):
        """Every user of [u_begin, u_end): the whole history against every item, in batches; device time (ms),
        users scored, similarity entries touched, finite scores."""
        B = max(1, min(args.score_batch, max(u_end - u_begin, 1)))
        row_len = (st.sim_indptr[1:] - st.sim_indptr[:-1]).cpu().numpy()
        a_lo, a_hi = int(R.indptr[u_begin]), int(R.indptr[u_end])
        d_ri = torch.from_numpy(R.indices[a_lo:a_hi].astype(np.int32)).to(dev)
        d_rv = torch.from_numpy((R.data[a_lo:a_hi] - means[R.indices[a_lo:a_hi]]).astype(np.float32)).to(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        total_ms, scored, touched, finite = 0.0, 0, 0, 0
        for u0 in range(u_begin, u_end, B):
            u1 = min(u0 + B, u_end)
            a0, a1 = int(R.indptr[u0]) - a_lo, int(R.indptr[u1]) - a_lo
            ref_ptr = torch.from_numpy((R.indptr[u0 : u1 + 1] - R.indptr[u0]).astype(np.int64)).to(dev)
            if u0 == u_begin:  # warm-up launch
                st.score_all_items(ref_ptr, d_ri[a0:a1], d_rv[a0:a1], KNN_MAX_NBRS, 1)
            e0.record()
            sc, ct = st.score_all_items(ref_ptr, d_ri[a0:a1], d_rv[a0:a1], KNN_MAX_NBRS, 1)
            e1.record()
            torch.cuda.synchronize()
            if dumped is not None and rank == 0 and u1 == u_end:  # the last launch: a fixed sample of its queries
                rows = sample_rows(u1 - u0, 32, 3)
                dumped["knn_score_users"] = (u0 + rows).astype(np.float64)
                d_rows = torch.from_numpy(rows).to(dev)
                # an item without enough neighbours has no score (NaN): 0 there, and the mask says which are scored
                scores = sc.index_select(0, d_rows).cpu().numpy()
                has_score = ~np.isnan(scores)
                dumped["knn_score_scores"] = np.where(has_score, scores, np.float32(0.0))
                dumped["knn_score_scored"] = has_score.astype(np.float32)
                dumped["knn_score_counts"] = ct.index_select(0, d_rows).cpu().numpy().astype(np.float32)
            total_ms += e0.elapsed_time(e1)
            scored += u1 - u0
            touched += int(row_len[R.indices[a_lo + a0 : a_lo + a1]].sum())
            finite += int(torch.isfinite(sc).sum().item())
            del sc, ct
        return total_ms, scored, touched, finite

    def check_parity(indptr, cols, vals, extra: dict | None = None):
        if args.no_parity or rank != 0:
            return
        from oracle import parity as par

        rows = par.sample_knn_rows(cost, np.diff(kiu.indptr), seed=3)
        r = par.check_knn_rows(kui, kiu, rows, indptr.cpu().numpy(), cols.cpu().numpy(), vals.cpu().numpy(),
                               KNN_MIN_SIM, KNN_SAVE)  # fmt: skip
        r["hottest_item_products"] = int(cost.max())
        if extra:
            r.update(extra)
            r["ok"] = bool(r["ok"] and all(v for v in extra.values() if isinstance(v, bool)))
        parity["knn_exact"] = r
        log(f"[bench] parity kNN: {r['rows']} sampled rows ({r['neighbours_compared']} neighbours), "
            f"mismatched {r['n_mismatched']} ok={r['ok']}")

    if world > 1:
        # item-sharded build: UI replicated, rows dealt by cost, one exchange of the top-K rows
        import torch.distributed as dist

        from lkpy_b200.parallel import sharded_knn_build_topk

        def sbuild():
            plan.prepare()  # tile pointers, costs, units: part of the build, as at N = 1
            return sharded_knn_build_topk(plan, KNN_MIN_SIM, KNN_SAVE)

        sbuild()
        dist.barrier()
        torch.cuda.synchronize()
        reps = args.steps
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(reps):
            cols, vals, cnt = sbuild()
        s1.record()
        dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([s0.elapsed_time(s1) / reps], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        extra = None
        if dumped is not None and rank == 0:
            dump_csr(dumped, "knn_sim", *engine.topk_rows_to_csr(cols, vals, cnt))
        if not args.no_parity:
            from oracle import parity as par

            live = torch.arange(cols.shape[1], device=dev)[None, :] < cnt[:, None]  # padding past a row's count is not data
            cs = par.checksum(torch.where(live, cols, 0).cpu().numpy(), torch.where(live, vals, 0.0).cpu().numpy(),
                              cnt.cpu().numpy())
            tt = torch.tensor([cs >> 32, cs & 0xFFFFFFFF], dtype=torch.int64, device=dev)
            lo, hi = tt.clone(), tt.clone()
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            extra = {"result_equal_across_ranks": bool(torch.equal(lo, hi))}
        # scoring shards by user (SURVEY.md §8e): the similarity matrix is replicated after the build, every rank
        # scores a contiguous user range balanced by history length; no collective on the data path
        from lkpy_b200.parallel import row_bounds_by_nnz

        dist.barrier()
        local = torch.zeros(4, device=dev, dtype=torch.float64)  # ok, ms, users, finite scores
        err = ""
        try:  # no collective inside: a rank that fails here still reaches the reductions below
            R = inter.coo().tocsr()
            n_score = inter.n_users if args.score_users <= 0 else min(args.score_users, inter.n_users)
            bounds = row_bounds_by_nnz(R.indptr[: n_score + 1], world)
            st = engine.KnnScorerState.create(inter.n_items, *engine.topk_rows_to_csr(cols, vals, cnt), dev)
            s_ms, scored, _touched, finite = score_users(st, R, int(bounds[rank]), int(bounds[rank + 1]))
            local = torch.tensor([1.0, s_ms, float(scored), float(finite)], device=dev, dtype=torch.float64)
            del st
        except Exception as e:  # the scoring line must not take the build line (and the ALS headline) down with it
            err = f"{type(e).__name__}: {e}"
        mn, mx, sm = local.clone(), local.clone(), local.clone()
        dist.all_reduce(mn, op=dist.ReduceOp.MIN)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        if float(mn[0].item()) == 1.0:
            score = {
                "users": int(sm[2].item()), "targets_per_user": inter.n_items, "ms": float(mx[1].item()),
                "users_per_s": float(sm[2].item()) / (float(mx[1].item()) * 1e-3),
                "scored_fraction": float(sm[3].item()) / max(float(sm[2].item()) * inter.n_items, 1.0),
                "parallelism": f"users sharded by history length over {world} GPUs, similarity matrix replicated; "
                               "time = max over ranks of the summed device time of the rank's launches",
            }  # fmt: skip
        else:
            score = {"error": err or "a rank failed"}
        if rank != 0:
            return None
        check_parity(*engine.topk_rows_to_csr(cols, vals, cnt), extra=extra)
        log(f"[bench] kNN build x{world}: {ms:.1f} ms = {inter.n_items / (ms * 1e-3):.0f} items/s; score {score}")
        return {
            "workload": "ML-25M-shaped synthetic ItemKNNScorer explicit, min_sim=1e-6, save_nbrs=20 (BASELINE configs[2])",
            "build_ms": ms, "build_items_per_s": inter.n_items / (ms * 1e-3),
            "neighbours_kept": int(cnt.sum().item()), "parallelism": f"item rows dealt by cost over {world} GPUs",
            "score": score,
        }  # fmt: skip

    def build():
        # the whole build from the resident CSR inputs: tile pointers, row costs, work order,
        # accumulate + top-K, merge, compaction to CSR
        plan.prepare()
        cols, vals, cnt = plan.build_topk(KNN_MIN_SIM, KNN_SAVE)
        return plan, engine.topk_rows_to_csr(cols, vals, cnt)

    plan, csr = build()  # warm-up (also loads the kernels)
    torch.cuda.synchronize()
    reps = args.steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        plan, csr = build()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    if dumped is not None:
        dump_csr(dumped, "knn_sim", *csr)
    # the accumulate kernel alone (same stream, events around the launch)
    import ctypes as C

    from lkpy_b200 import _lib

    u = plan.units(split_hot=True)
    part_cols = torch.empty(u["n_units"] * KNN_SAVE, dtype=torch.int32, device=dev)
    part_vals = torch.empty(u["n_units"] * KNN_SAVE, dtype=torch.float32, device=dev)
    part_cnt = torch.zeros(u["n_units"], dtype=torch.int32, device=dev)
    a = plan._args(u, u["sched"], KNN_MIN_SIM, KNN_SAVE)
    a.d_part_cols, a.d_part_vals, a.d_part_cnt = _lib.ptr(part_cols), _lib.ptr(part_vals), _lib.ptr(part_cnt)
    k0.record()
    _lib.check(_lib.lib().lk_knn_build(C.byref(a), _lib.stream_ptr()), "lk_knn_build")
    k1.record()
    torch.cuda.synchronize()
    kms = k0.elapsed_time(k1)
    del part_cols, part_vals, part_cnt
    nnz_out = int(csr[0][-1].item())
    alg = knn_build_bytes(products, inter.nnz, inter.n_users, inter.n_items, nnz_out)
    achieved = alg / (kms * 1e-3) / 1e9
    out = {
        "workload": "ML-25M-shaped synthetic ItemKNNScorer explicit, min_sim=1e-6, save_nbrs=20 (BASELINE configs[2])",
        "build_ms": ms,
        "build_items_per_s": inter.n_items / (ms * 1e-3),
        "build_kernel_ms": kms,
        "products": products,
        "neighbours_kept": nnz_out,
        "geometry": {"warps": plan.geom.warps, "tile_cols": plan.geom.tile_cols, "halves": plan.geom.n_halves,
                     "ctas_per_sm": plan.geom.ctas_per_sm, "work_units": u["n_units"]},
        "roofline": {"bound": "hbm", "kernel": "knn_build_kernel", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak,
                     "traffic": ncu_traffic("knn_build_kernel_bytes", world), "algorithmic_bytes": alg,
                     "peak_source": peak_src},
        "_kui": kui, "_kiu": kiu, "_cost": cost,
    }  # fmt: skip
    log(f"[bench] kNN build: {ms:.1f} ms = {out['build_items_per_s']:.0f} items/s; accumulate kernel {kms:.1f} ms, "
        f"{achieved:.0f} GB/s algorithmic = {achieved / peak:.3f} of peak")
    check_parity(*csr)

    # ---- end to end through the plugin call: host CSR in -> host CSR out (item_train.rs:32-93)
    if not args.profile:
        accel.clear_cache()
        accel.run_accel_task(accel.compute_similarities(kui, kiu, (inter.n_users, inter.n_items), KNN_MIN_SIM, KNN_SAVE))
        ts = []
        for _ in range(3):
            accel.clear_cache()  # the device copies of the operands are part of the call
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = accel.run_accel_task(
                accel.compute_similarities(kui, kiu, (inter.n_users, inter.n_items), KNN_MIN_SIM, KNN_SAVE)
            )
            ts.append(time.perf_counter() - t0)
        e2e_s = float(np.median(ts))
        h2d = int(sum(m.indptr.nbytes + m.indices.nbytes + m.values.nbytes for m in (kui, kiu)))
        d2h = int(sum(r.nbytes for r in res))  # LargeList chunks: offsets + index + value buffers
        out["e2e"] = {
            "value": inter.n_items / e2e_s, "unit": "items/s", "ms": e2e_s * 1e3, "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h,
            "api": "accel.compute_similarities via run_accel_task: host CSR (UI, IU) in, host LargeList-layout CSR out",
        }  # fmt: skip
        accel.clear_cache()
        # and through the component: ItemKNNScorer.train (host prep + upload + build + download)
        from lkpy_b200.knn import ItemKNNScorer

        m = ItemKNNScorer(max_nbrs=KNN_MAX_NBRS, min_sim=KNN_MIN_SIM, save_nbrs=KNN_SAVE)
        t0 = time.perf_counter()
        m.train(Dataset(inter))
        torch.cuda.synchronize()
        out["train_e2e_ms"] = (time.perf_counter() - t0) * 1e3
        out["train_prep"] = m.__dict__.get("prep_where", "host (SciPy)")
        del m
        log(f"[bench] kNN e2e: compute_similarities {e2e_s * 1e3:.0f} ms = {out['e2e']['value']:.0f} items/s; "
            f"ItemKNNScorer.train {out['train_e2e_ms']:.0f} ms ({out['train_prep']} prep)")

    # ---- scoring: every user's history against every item, in batches
    indptr, c, v = csr
    st = engine.KnnScorerState.create(inter.n_items, indptr, c, v, dev)
    R = inter.coo().tocsr()
    n_score = inter.n_users if args.score_users <= 0 else min(args.score_users, inter.n_users)
    B = max(1, min(args.score_batch, n_score))
    try:
        try:
            total_ms, scored, touched, finite = score_users(st, R, 0, n_score)
        except (torch.OutOfMemoryError, RuntimeError) as e:
            # the wide default batch is a throughput choice, not a requirement: fall back to the batch the round's
            # measurements were taken with rather than lose the line
            log(f"[bench] kNN score at {B} users per launch failed ({type(e).__name__}: {e}); retrying at 4096")
            torch.cuda.empty_cache()
            args.score_batch = B = min(4096, n_score)
            total_ms, scored, touched, finite = score_users(st, R, 0, n_score)
        alg_s = knn_score_bytes(touched, int(R.indptr[n_score]), scored * inter.n_items)
        ach_s = alg_s / (total_ms * 1e-3) / 1e9
        out["score"] = {
            "users": scored, "targets_per_user": inter.n_items, "batch": B, "ms": total_ms,
            "users_per_s": scored / (total_ms * 1e-3), "scored_fraction": finite / max(scored * inter.n_items, 1),
            "roofline": {"bound": "hbm", "kernel": "knn_score_dense_kernel", "achieved": ach_s, "peak": peak, "unit": "GB/s",
                         "frac": ach_s / peak, "traffic": ncu_traffic("knn_score_dense_kernel_v3_bytes_per_2048_users", world),
                         "traffic_note": "per launch of 2,048 users (the ncu capture), not per launch of this run",
                         "algorithmic_bytes": alg_s, "peak_source": peak_src},
        }  # fmt: skip
        out["build_plus_score_s"] = ms * 1e-3 + total_ms * 1e-3 * (inter.n_users / max(scored, 1))
        log(f"[bench] kNN score: {scored} users x all items in {total_ms:.1f} ms = {out['score']['users_per_s']:.0f} users/s, "
            f"{ach_s:.0f} GB/s algorithmic = {ach_s / peak:.3f} of peak")
    except Exception as e:  # the scoring line must not take the build line (and the ALS headline) down with it
        out["score"] = {"error": f"{type(e).__name__}: {e}"}
        log(f"[bench] kNN score failed: {out['score']['error']}")
    return out


if __name__ == "__main__":
    main()
