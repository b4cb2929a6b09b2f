"""
Generator harness: the reference's OWN Python classes for the hot path — ``lenskit.training``,
``lenskit.pipeline.components.Component``, ``lenskit.data.matrix.SparseRowArray``, ``ItemList``, ``Vocabulary``,
``RecQuery``, ``basic.bias.BiasModel``, ``lenskit.als._common / _implicit / _explicit``, ``lenskit.knn.item / user`` —
loaded file by file from a lenskit source checkout (``set_root``), with ``lenskit._accel`` bound to
``lkpy_b200.accel`` exactly as INTEGRATION.md §1 describes.  ``make_reference_classes.py`` runs the reference's
classes through it and stores what they pass to and get back from the accelerator API; the tests replay that
record and never load the reference.

The reference package cannot be imported as a whole (its ``__init__`` needs ``lazy_loader`` /
``structlog``, its data layer needs the Rust extension's ``IDIndex`` / ``CoordinateTable``), so the modules
the hot path does not touch are replaced by small fakes: logging, the thread-pool configuration (the task
runner itself, ``parallel/_task.py``, is the reference's), Python stand-ins for
the Rust helpers of the data model (``IDIndex``, ``scatter_array`` ...), and the slice of ``Dataset`` the two
trainers read (``Dataset.interactions().matrix().scipy(...)``, the vocabularies).
Everything between the user's ``scorer.train(dataset)`` and the accelerator call is the reference's code.
"""

from __future__ import annotations

import contextlib
import importlib.util
import sys
import types
from pathlib import Path

import numpy as np
from scipy.sparse import coo_array

REF_SRC = Path("src/lenskit")


def set_root(checkout: Path) -> None:
    """Point the sandbox at a lenskit source checkout (the directory holding ``src/lenskit``)."""
    global REF_SRC
    REF_SRC = Path(checkout) / "src" / "lenskit"
    if not (REF_SRC / "als" / "_implicit.py").exists():
        raise FileNotFoundError(f"no lenskit sources under {REF_SRC}")


# ---------------------------------------------------------------------------
# fakes for what the hot path does not touch
# ---------------------------------------------------------------------------


class _Log:
    """structlog-shaped no-op logger."""

    def bind(self, **_kw):
        return self

    def _noop(self, *_a, **_kw):
        return None

    debug = info = warning = warn = error = trace = _noop


class _Stopwatch:
    def __str__(self):
        return "0s"


class _AtomicInt:
    """``_accel.AtomicInt`` as parallel/_task.py uses it (thread names)."""

    def __init__(self):
        self._v = 0

    def fetch_add(self, n: int = 1) -> int:
        v, self._v = self._v, self._v + n
        return v


class _NestedPool:
    @staticmethod
    def active_accel_pool():
        return None


class _Progress:
    def __init__(self, *_a, **_kw):
        self.updates = 0

    def update(self, *_a, **_kw):
        self.updates += 1

    def __enter__(self):
        return self

    def __exit__(self, *_a):
        return False


class _MatrixView:
    """``data.interactions().matrix()``: the one call the trainers make on it."""

    def __init__(self, inter):
        self._inter = inter

    def scipy(self, attribute: str | None = None, layout: str = "csr", **_kw):
        it = self._inter
        vals = it.ratings.astype(np.float32) if attribute == "rating" else np.ones(it.nnz, dtype=np.float32)
        m = coo_array((vals, (it.users, it.items)), shape=(it.n_users, it.n_items))
        return m if layout == "coo" else m.tocsr()


class _Relationship:
    def __init__(self, inter):
        self._inter = inter

    def matrix(self, **_kw):
        return _MatrixView(self._inter)


class FakeDataset:
    """The slice of ``lenskit.data.Dataset`` the ALS / kNN trainers read, over ``lkpy_b200.data.Interactions``."""

    def __init__(self, inter):
        Vocabulary = sys.modules["lenskit.data"].Vocabulary  # the reference's own class (data/_vocab.py)

        self._inter = inter
        self.users = Vocabulary(inter.user_ids if inter.user_ids is not None else np.arange(inter.n_users), "user")
        self.items = Vocabulary(inter.item_ids if inter.item_ids is not None else np.arange(inter.n_items), "item")

    user_count = property(lambda self: self._inter.n_users)
    item_count = property(lambda self: self._inter.n_items)
    interaction_count = property(lambda self: self._inter.nnz)

    def interaction_matrix(self, *, format: str = "scipy", layout: str = "csr", field: str | None = None, **_kw):
        assert format == "scipy"
        return _MatrixView(self._inter).scipy(field, layout=layout)

    def interactions(self, *_a, **_kw):
        return _Relationship(self._inter)


class IDIndex:
    """Python stand-in for the Rust ``_accel.data.IDIndex`` (src/accel/data/index.rs:97-139) behind the
    reference's real ``Vocabulary`` / ``ItemList``: id -> position; unknown (or wrongly typed) ids give None /
    null."""

    def __init__(self, ids=None):
        import pyarrow as pa

        self._ids = pa.array([], type=pa.int64()) if ids is None else (ids if isinstance(ids, pa.Array) else pa.array(ids))
        self._pos = {v: i for i, v in enumerate(self._ids.to_pylist())}

    def get_index(self, id_):
        try:
            if isinstance(id_, np.generic):
                id_ = id_.item()
            return self._pos.get(id_)
        except TypeError:
            return None

    def get_indexes(self, ids):
        import pyarrow as pa

        vals = ids.to_pylist() if isinstance(ids, (pa.Array, pa.ChunkedArray)) else list(np.asarray(ids).tolist())
        return pa.array([None if v is None else self._pos.get(v) for v in vals], type=pa.int32())

    def id_array(self):
        return self._ids

    def __len__(self) -> int:
        return len(self._ids)


def _data_shims() -> types.SimpleNamespace:
    """``lenskit._accel.data`` as far as ``data/_vocab.py``, ``_items.py`` and ``_mtarray.py`` use it."""
    import hashlib

    import pyarrow as pa

    def hash_array(arr) -> str:
        return hashlib.md5(repr(arr.to_pylist()).encode()).hexdigest()

    def argsort_descending(scores):
        v = scores.to_numpy(zero_copy_only=False).astype(np.float64)
        order = np.argsort(-np.where(np.isnan(v), -np.inf, v), kind="stable")
        return pa.array(order[~np.isnan(v[order])].astype(np.int32))

    def argtopn(scores, n: int):  # the step after the scorers (SURVEY.md §8f N2): this package's mirror
        from lkpy_b200 import accel

        return accel.argtopn(scores, n)

    def scatter_array_empty(dst_size: int, idx, src):
        out = [None] * int(dst_size)
        for i, v in zip(idx.to_pylist(), src.to_pylist()):
            if i is not None:
                out[i] = v
        return pa.array(out, type=src.type)

    def scatter_array(dst, idx, src):
        out = dst.to_pylist()
        for i, v in zip(idx.to_pylist(), src.to_pylist()):
            if i is not None:
                out[i] = v
        return pa.array(out, type=dst.type)

    return types.SimpleNamespace(IDIndex=IDIndex, hash_array=hash_array, argsort_descending=argsort_descending,
                                 argtopn=argtopn, scatter_array=scatter_array, scatter_array_empty=scatter_array_empty)  # fmt: skip


def _module(name: str, package: bool = False, **attrs) -> types.ModuleType:
    m = types.ModuleType(name)
    if package:
        m.__path__ = []  # a package without files: submodules are registered by hand
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


def _load(name: str, rel: str) -> types.ModuleType:
    spec = importlib.util.spec_from_file_location(name, REF_SRC / rel)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    parent, _, leaf = name.rpartition(".")
    if parent in sys.modules:
        setattr(sys.modules[parent], leaf, mod)
    return mod


@contextlib.contextmanager
def reference_modules():
    """Install the sandbox in ``sys.modules`` and yield ``{module name: module}``; removed again on exit."""
    from lkpy_b200 import accel

    def ours(name):  # nothing of a real lenskit install may leak in or out
        return name == "lenskit" or name.startswith("lenskit.") or name in ("structlog", "structlog.stdlib")

    saved = {k: v for k, v in sys.modules.items() if ours(k)}
    for k in saved:
        del sys.modules[k]
    try:
        _module("structlog", package=True, stdlib=_module("structlog.stdlib", BoundLogger=object))
        _module("lenskit", package=True)
        _module("lenskit.logging", package=True, get_logger=lambda *_a, **_k: _Log(), item_progress=_Progress,
                Progress=_Progress, Stopwatch=_Stopwatch, trace=lambda *_a, **_k: None)  # fmt: skip
        _module("lenskit.logging._resource", cur_memory=lambda: "0", max_memory=lambda: "0")
        par = _module("lenskit.parallel", package=True, ensure_parallel_init=lambda: None,
                      is_free_threaded=lambda: False)  # fmt: skip
        _module("lenskit.parallel.config", ensure_parallel_init=lambda: None)
        _module("lenskit.parallel._pool", NestedPool=_NestedPool)
        # INTEGRATION.md §1: the module the reference imports its kernels from — als and knn are this package's;
        # `data` (the Rust helpers of the reference's data model, outside the hot path) is a Python stand-in
        sys.modules["lenskit"]._accel = _module("lenskit._accel", package=True, als=accel.als, knn=accel.knn,
                                                data=_data_shims(), AtomicInt=_AtomicInt,
                                                NestedAccelPool=object)  # fmt: skip
        # the reference's own task runner (parallel/_task.py:25-135) drives this package's AccelTask objects
        par.run_accel_task = _load("lenskit.parallel._task", "parallel/_task.py").run_accel_task
        from typing import Literal

        _module("lenskit.data", package=True, Dataset=FakeDataset, FeedbackType=Literal["explicit", "implicit"])
        for pkg in ("lenskit.config", "lenskit.math", "lenskit.pipeline", "lenskit.als", "lenskit.knn", "lenskit.basic"):
            _module(pkg, package=True)
        mods = {}
        for name, rel in (
            ("lenskit.diagnostics", "diagnostics.py"),
            ("lenskit.lazy", "lazy.py"),
            ("lenskit.torch", "torch.py"),
            ("lenskit.data.types", "data/types.py"),
            ("lenskit.data.matrix", "data/matrix.py"),
            ("lenskit.data._checks", "data/_checks.py"),
            ("lenskit.data._mtarray", "data/_mtarray.py"),
            ("lenskit.data._arrow", "data/_arrow.py"),
            ("lenskit.data._vocab", "data/_vocab.py"),
            ("lenskit.data._items", "data/_items.py"),
            ("lenskit.data._query", "data/_query.py"),
            ("lenskit.config.common", "config/common.py"),
            ("lenskit.math.solve", "math/solve.py"),
            ("lenskit.random", "random.py"),
            ("lenskit.pipeline._types", "pipeline/_types.py"),
            ("lenskit.pipeline.components", "pipeline/components.py"),
        ):
            mods[name] = _load(name, rel)
        sys.modules["lenskit.pipeline"].Component = mods["lenskit.pipeline.components"].Component
        dpk = sys.modules["lenskit.data"]
        dpk.Vocabulary, dpk.ItemList = mods["lenskit.data._vocab"].Vocabulary, mods["lenskit.data._items"].ItemList
        dpk.RecQuery, dpk.QueryInput = mods["lenskit.data._query"].RecQuery, mods["lenskit.data._query"].QueryInput
        dpk.ID = mods["lenskit.data.types"].ID
        for name, rel in (
            ("lenskit.training", "training.py"),
            ("lenskit.basic.bias", "basic/bias.py"),
        ):
            mods[name] = _load(name, rel)
        sys.modules["lenskit.basic"].BiasModel = mods["lenskit.basic.bias"].BiasModel
        sys.modules["lenskit.basic"].Damping = mods["lenskit.basic.bias"].Damping
        for name, rel in (
            ("lenskit.als._common", "als/_common.py"),
            ("lenskit.als._implicit", "als/_implicit.py"),
            ("lenskit.als._explicit", "als/_explicit.py"),
            ("lenskit.knn.item", "knn/item.py"),
            ("lenskit.knn.user", "knn/user.py"),
        ):
            mods[name] = _load(name, rel)
        yield mods
    finally:
        import pyarrow as pa

        for ext in ("lenskit.sparse_index", "lenskit.sparse_index_list", "lenskit.sparse_row"):
            with contextlib.suppress(Exception):  # registered by data/matrix.py when it was loaded
                pa.unregister_extension_type(ext)
        for k in [k for k in sys.modules if ours(k)]:
            del sys.modules[k]
        sys.modules.update(saved)
