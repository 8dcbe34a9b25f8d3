"""``HNSW`` -- search-only B200 counterpart of ``pecos.ann.hnsw.HNSW``.

The class keeps the reference's public surface for the load / search path, so code written against
``pecos.ann.hnsw.HNSW`` (pecos/ann/hnsw/model.py) runs unchanged:

=============================================  =======================================================
``HNSW.load(model_folder, lazy_load=False)``   reads ``param.json`` + ``c_model/`` written by the reference
``HNSW.predict(X, pred_params, searchers,      top-k neighbours per row of ``X``; CSR (distances as values) or a pair of
ret_csr=True)``                                ``(indices, distances)`` arrays
``HNSW.PredParams(efS, topk, threads)``        search parameters (``threads`` is accepted and ignored: the GPU kernel
                                               assigns one warp per query)
``HNSW.searchers_create(n)`` / ``Searchers``   opaque scratch token (the per-warp scratch lives with the engine)
=============================================  =======================================================

Index construction stays on the reference CPU library; both index kinds can also be built on the GPU by
``pecos_b200.hnsw_build.build_hnsw_index`` (dense rows: tiled GEMMs; ``scipy.sparse`` rows: the exact sparse kernels of
``csrc/hnsw_build_sparse.cu``), which writes files that this class and the reference both load.  Served index kinds: dense ``drm`` and sparse ``csr`` float32 with the ``ip`` or ``l2`` metric
(csr rows: column indices strictly ascending -- queries are canonicalised with ``sum_duplicates()`` / ``sort_indices()``
when needed).  There is no CPU fallback: loading without a visible CUDA device raises ``RuntimeError``.
"""
import dataclasses as dc
import json
import os
from ctypes import POINTER, byref, c_bool, c_char_p, c_float, c_uint32, c_void_p

import numpy as np
import scipy.sparse as smat

from .core import ScipyCsrF32, ScipyDrmF32, get_clib

_REQUIRED_KEYS = ("model", "data_type", "metric_type", "num_item", "feat_dim")


def _read_index_meta(model_folder):
    """``param.json`` of a saved index -> dict; validates what the loader relies on."""
    path = os.path.join(model_folder, "param.json")
    with open(path, "r", encoding="utf-8") as f:
        meta = json.load(f)
    missing = [k for k in _REQUIRED_KEYS if k not in meta]
    if missing:
        raise ValueError(f"{path}: missing field(s) {missing}")
    if meta["model"] != "HNSW":
        raise ValueError(f"{path}: model = {meta['model']!r}, expected 'HNSW'")
    return meta


class HNSW(object):
    @dc.dataclass
    class PredParams(object):
        efS: int = 100
        topk: int = 10
        threads: int = 1

        @classmethod
        def from_dict(cls, d):
            known = {f.name for f in dc.fields(cls)}
            return cls(**{k: int(v) for k, v in (d or {}).items() if k in known})

    class Searchers(object):
        """Owner of the native searcher token; released with the object."""

        def __init__(self, model, num_searcher=1):
            self._release = model.fn_dict["searchers_destruct"]
            self.searchers_ptr = c_void_p(model.fn_dict["searchers_create"](model.model_ptr, int(num_searcher)))

        def ctypes(self):
            return self.searchers_ptr

        def __del__(self):
            ptr, self.searchers_ptr = getattr(self, "searchers_ptr", None), None
            if ptr:
                try:
                    self._release(ptr)
                except Exception:
                    pass

    def __init__(self, model_ptr, num_item, feat_dim, fn_dict, pred_params=None, data_type="drm", metric_type="ip"):
        self.model_ptr, self.fn_dict = model_ptr, fn_dict
        self.num_item, self.feat_dim = int(num_item), int(feat_dim)
        self.pred_params = pred_params if pred_params is not None else self.PredParams()
        self._data_type, self._metric_type = data_type, metric_type

    data_type = property(lambda self: self._data_type)
    metric_type = property(lambda self: self._metric_type)

    def __del__(self):
        ptr, self.model_ptr = getattr(self, "model_ptr", None), None
        if ptr and getattr(self, "fn_dict", None):
            try:
                self.fn_dict["destruct"](ptr)
            except Exception:
                pass

    # ------------------------------------------------------------------ load
    @classmethod
    def load(cls, model_folder, lazy_load=False):
        meta = _read_index_meta(model_folder)
        native_dir = os.path.join(model_folder, "c_model")
        if not os.path.isdir(native_dir):
            raise ValueError(f"{native_dir} is not a directory: not a saved HNSW index")
        lib = get_clib()
        symbols = lib.ann_hnsw_init(meta["data_type"], meta["metric_type"])  # raises for index kinds this engine does not serve
        lib.require_gpu()
        handle = symbols["load"](c_char_p(native_dir.encode("utf-8")), c_bool(bool(lazy_load)))
        return cls(c_void_p(handle), meta["num_item"], meta["feat_dim"], symbols,
                   cls.PredParams.from_dict(meta.get("pred_kwargs")), meta["data_type"], meta["metric_type"])

    def get_pred_params(self):
        return dc.replace(self.pred_params)

    def searchers_create(self, num_searcher=1):
        if not self.model_ptr:
            raise ValueError("the index is not loaded")
        if int(num_searcher) < 1:
            raise ValueError(f"num_searcher must be >= 1, got {num_searcher}")
        return HNSW.Searchers(self, num_searcher)

    # ------------------------------------------------------------------ search
    @staticmethod
    def create_pymat(X):
        """Query matrix -> (ctypes view, kind): dense float32 row-major, or csr float32 with ascending column indices."""
        if isinstance(X, ScipyDrmF32):
            return X, "drm"
        if isinstance(X, ScipyCsrF32):
            return X, "csr"
        if isinstance(X, np.ndarray):
            return ScipyDrmF32.init_from(np.ascontiguousarray(X, dtype=np.float32)), "drm"
        if smat.issparse(X):
            X = smat.csr_matrix(X, dtype=np.float32)
            if not X.has_canonical_format:  # the intersection kernels walk strictly ascending indices
                X = X.copy()
                X.sum_duplicates()
            return ScipyCsrF32.init_from(X), "csr"
        raise ValueError(f"queries of type {type(X)} are not supported")

    def predict(self, X, pred_params=None, searchers=None, ret_csr=True):
        params = pred_params if pred_params is not None else self.get_pred_params()
        view, kind = self.create_pymat(X)
        if kind != self.data_type:
            raise ValueError(f"{kind} queries cannot be searched in a {self.data_type} index")
        if view.cols != self.feat_dim:
            raise ValueError(f"query dimension {view.cols} != index dimension {self.feat_dim}")
        n, k = int(view.rows), int(params.topk)
        # the native call only fills the slots it found neighbours for; the rest must read as zeros (reference contract)
        idx = np.zeros((n, k), dtype=np.uint32)
        dist = np.zeros((n, k), dtype=np.float32)
        token = searchers.ctypes() if searchers is not None else None
        self.fn_dict["predict"](self.model_ptr, byref(view), idx.ctypes.data_as(POINTER(c_uint32)),
                                dist.ctypes.data_as(POINTER(c_float)), int(params.efS), k, int(params.threads), token)
        if not ret_csr:
            return idx, dist
        row_starts = np.arange(n + 1, dtype=np.int64) * k
        return smat.csr_matrix((dist.ravel(), idx.ravel().astype(np.int64), row_starts), shape=(n, self.num_item), dtype=np.float32)
