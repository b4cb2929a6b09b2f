"""Shared helpers for the parity tests."""

from __future__ import annotations

import threading
import time

import numpy as np

from lkpy_b200 import data


def implicit_init(rng: np.random.Generator, n_items: int, n_users: int, k: int):
    """Reference init: items first, then users; (0.01*N(0,1))^2 (als/_implicit.py:152-155)."""

    def one(n):
        m = rng.standard_normal((n, k), dtype=np.float32) * 0.01
        m *= m
        return m

    q = one(n_items)
    p = one(n_users)
    return p, q


def explicit_init(rng: np.random.Generator, n_items: int, n_users: int, k: int):
    """Reference init: unit-norm random rows (als/_explicit.py:105-108)."""

    def one(n):
        m = rng.standard_normal((n, k), dtype=np.float32)
        m /= np.linalg.norm(m, axis=1).reshape((n, 1))
        return m

    q = one(n_items)
    p = one(n_users)
    return p, q


def rel_fro(a: np.ndarray, b: np.ndarray) -> float:
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def small_synth(n_users=600, n_items=400, nnz=20000, seed=7, ratings=True):
    return data.synth_interactions(n_users, n_items, nnz, seed, ratings=ratings)


def sha256(a: np.ndarray) -> str:
    """Digest of an array's bytes (dtype and shape are the caller's to check)."""
    import hashlib

    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def csr_digest(m) -> str:
    """One digest over a CSR matrix: shape, int64 offsets, int32 columns, float32 value bits."""
    return sha256(np.concatenate([
        np.asarray(m.shape, dtype=np.int64).view(np.uint8), np.asarray(m.indptr, dtype=np.int64).view(np.uint8),
        np.asarray(m.indices, dtype=np.int32).view(np.uint8), np.asarray(m.values, dtype=np.float32).view(np.uint8),
    ]))  # fmt: skip


def oracle_accel(monkeypatch) -> None:
    """No GPU: keep the accelerator entry points' own argument handling (Arrow ingest, the task protocol, the
    in-place contract on ``this``, the result layout) and swap only their device part for the CPU oracle."""
    import scipy.sparse as sps
    import torch

    import oracle
    from lkpy_b200 import accel

    def als_task(mode, matrix, this, other, otor, reg):
        this = accel._check_factor("this", this, writable=True)
        other = accel._check_factor("other", other)
        csr = accel.as_host_csr(matrix)
        assert csr.shape == (this.shape[0], other.shape[0])

        def run(_task):
            if mode == accel._lib.LK_ALS_IMPLICIT:
                new, delta = oracle.als_half("implicit", csr, this, other, otor_mat=otor)
            else:
                new, delta = oracle.als_half("explicit", csr, this, other, reg=reg)
            this[...] = new  # in place, like implicit.rs:57-64
            return float(delta)

        return accel.AccelTask(run, total=this.shape[0])

    def compute_similarities(ui_ratings, iu_ratings, shape, min_sim, save_nbrs):
        nu, ni = shape
        ui, iu = accel.as_host_csr(ui_ratings, ni), accel.as_host_csr(iu_ratings, nu)
        assert ui.shape == (nu, ni) and iu.shape == (ni, nu)

        def run(_task):
            S = oracle.knn_build(ui, iu, min_sim, save_nbrs)
            out = data.InteractionCSR(S.indptr.astype(np.int64), S.indices, S.data, (ni, ni))
            return accel.csr_to_arrow_chunks(out, 2000)

        return accel.AccelTask(run, total=ni)

    class CpuScorerState:
        """``engine.KnnScorerState`` with the oracle behind ``score``: accel._score runs unchanged around it."""

        def __init__(self, n_items, indptr, cols, vals, user_mode):
            n_rows = len(indptr) - 1
            self.explicit = vals is not None
            v = np.asarray(vals) if vals is not None else np.ones(len(cols), np.float32)
            self.S = sps.csr_array((v, np.asarray(cols), np.asarray(indptr)), shape=(n_rows, n_items))
            self.user_mode = user_mode

        @classmethod
        def create(cls, n_items, indptr, cols, vals, _dev, user_mode=False):
            return cls(n_items, indptr, cols, vals, user_mode)

        def score(self, _ref_ptr, ref_items, ref_vals, _tgt_ptr, tgt_items, max_nbrs, min_nbrs):
            if self.user_mode:  # the "history" is the neighbour list and carries the weights (user_score.rs:21-98)
                sc, ct = oracle.user_score(self.S, ref_items.numpy(), ref_vals.numpy(), tgt_items.numpy(), max_nbrs,
                                           min_nbrs, explicit=self.explicit)  # fmt: skip
            else:
                sc, ct = oracle.knn_score(self.S, ref_items.numpy(), None if ref_vals is None else ref_vals.numpy(),
                                          tgt_items.numpy(), max_nbrs, min_nbrs)  # fmt: skip
            return torch.from_numpy(sc), torch.from_numpy(ct)

    def argtopn_batch(scores, n):
        return [oracle.argtopn(np.ascontiguousarray(row, dtype=np.float32), int(min(n, len(row)))) for row in np.asarray(scores)]

    monkeypatch.setattr(accel, "argtopn_batch", argtopn_batch)
    monkeypatch.setattr(accel, "_als_task", als_task)
    monkeypatch.setattr(accel.knn, "compute_similarities", compute_similarities)
    monkeypatch.setattr(accel._lib, "require_device", lambda: torch.device("cpu"))
    monkeypatch.setattr(accel.engine, "KnnScorerState", CpuScorerState)


class TaskProbe:
    """Stands in for an ``AccelTask`` under the reference's ``run_accel_task`` and notes what it is asked."""

    def __init__(self, result=None, error=None):
        self.log: list[str] = []
        self.result, self.error = result, error

    def invoke(self, **kw):
        self.log.append(f"invoke({','.join(f'{k}={v!r}' for k, v in sorted(kw.items()))}) on {threading.current_thread().name.split('-')[0]}")
        time.sleep(0.5)  # long enough for two polls of current_progress()
        if self.error:
            raise self.error
        return self.result

    def current_progress(self):
        if not self.log or self.log[-1] != "current_progress()":
            self.log.append("current_progress()")
        return (0, 10)

    def cancel(self):
        self.log.append("cancel()")
