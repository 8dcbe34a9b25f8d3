"""ctypes shim over ``libpecos_b200_float32.so`` -- the B200 counterpart of ``pecos.core.base.corelib``.

Mirrors, for the two hot paths only, the reference's Python-side FFI layer:

* buffer views ``ScipyCsrF32`` / ``ScipyDrmF32`` ........ pecos/core/base.py:219-310
* result allocator ``ScipyCompressedSparseAllocator`` .. pecos/core/base.py:407-478
* ``corelib.xlinear_*`` helpers ......................... pecos/core/base.py:990-1095
* ``corelib.link_ann_hnsw_methods`` / fn_dict ........... pecos/core/base.py:1865-1964

There is no CPU fallback: if the CUDA library is missing, or no GPU is visible when a model is loaded,
a ``RuntimeError`` is raised.
"""
import ctypes
import os
from ctypes import (
    CFUNCTYPE,
    POINTER,
    byref,
    c_bool,
    c_char_p,
    c_double,
    c_float,
    c_int,
    c_int32,
    c_size_t,
    c_uint32,
    c_uint64,
    c_void_p,
    cast,
)

import numpy as np
import scipy.sparse as smat

LIB_BASENAME = "libpecos_b200_float32.so"
LIB_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib")
LIB_PATH = os.path.join(LIB_DIR, LIB_BASENAME)

# pecos/core/base.py:49
XLINEAR_INFERENCE_MODEL_TYPES = {"CSC": 0, "HASH_CHUNKED": 1, "BINARY_SEARCH_CHUNKED": 2}


class ScipyCsrF32(ctypes.Structure):
    """C view of a float32 scipy CSR matrix (pecos/core/base.py:219-266)."""

    _fields_ = [
        ("rows", c_uint32),
        ("cols", c_uint32),
        ("indptr", POINTER(c_uint64)),
        ("indices", POINTER(c_uint32)),
        ("data", POINTER(c_float)),
    ]

    @classmethod
    def init_from(cls, A, pinned=None):
        if not isinstance(A, smat.csr_matrix):
            raise ValueError("type(A) = {} is not supported".format(type(A)))
        if A.dtype != np.float32:
            raise ValueError("A.dtype = {} is not float32".format(A.dtype))
        self = cls()
        # keep the converted arrays alive for the duration of the call (same as the reference's py_buf)
        self.py_buf = {
            "indptr": np.ascontiguousarray(A.indptr, dtype=np.uint64),
            "indices": np.ascontiguousarray(A.indices, dtype=np.uint32),
            "data": np.ascontiguousarray(A.data, dtype=np.float32),
        }
        self.rows, self.cols = A.shape
        self.indptr = self.py_buf["indptr"].ctypes.data_as(POINTER(c_uint64))
        self.indices = self.py_buf["indices"].ctypes.data_as(POINTER(c_uint32))
        self.data = self.py_buf["data"].ctypes.data_as(POINTER(c_float))
        return self

    @classmethod
    def init_from_arrays(cls, rows, cols, indptr, indices, data):
        """Wrap already-typed arrays (uint64/uint32/float32) without copying, e.g. pinned host buffers."""
        assert indptr.dtype == np.uint64 and indices.dtype == np.uint32 and data.dtype == np.float32
        self = cls()
        self.py_buf = {"indptr": indptr, "indices": indices, "data": data}
        self.rows, self.cols = rows, cols
        self.indptr = indptr.ctypes.data_as(POINTER(c_uint64))
        self.indices = indices.ctypes.data_as(POINTER(c_uint32))
        self.data = data.ctypes.data_as(POINTER(c_float))
        return self


class ScipyCscF32(ctypes.Structure):
    """C view of a float32 scipy CSC matrix (pecos/core/base.py:177-216); same layout as ScipyCsrF32 with col_ptr /
    row_idx in place of row_ptr / col_idx."""

    _fields_ = [
        ("rows", c_uint32),
        ("cols", c_uint32),
        ("indptr", POINTER(c_uint64)),
        ("indices", POINTER(c_uint32)),
        ("data", POINTER(c_float)),
    ]

    @classmethod
    def init_from(cls, A):
        if not isinstance(A, smat.csc_matrix):
            raise ValueError("type(A) = {} is not supported".format(type(A)))
        if A.dtype != np.float32:
            raise ValueError("A.dtype = {} is not float32".format(A.dtype))
        self = cls()
        self.py_buf = {
            "indptr": np.ascontiguousarray(A.indptr, dtype=np.uint64),
            "indices": np.ascontiguousarray(A.indices, dtype=np.uint32),
            "data": np.ascontiguousarray(A.data, dtype=np.float32),
        }
        self.rows, self.cols = A.shape
        self.indptr = self.py_buf["indptr"].ctypes.data_as(POINTER(c_uint64))
        self.indices = self.py_buf["indices"].ctypes.data_as(POINTER(c_uint32))
        self.data = self.py_buf["data"].ctypes.data_as(POINTER(c_float))
        return self


class ScipyDrmF32(ctypes.Structure):
    """C view of a C-contiguous float32 ndarray (pecos/core/base.py:269-310)."""

    _fields_ = [("rows", c_uint32), ("cols", c_uint32), ("val", POINTER(c_float))]

    @classmethod
    def init_from(cls, A):
        if not isinstance(A, np.ndarray):
            raise ValueError("type(A) = {} is not supported".format(type(A)))
        if A.dtype != np.float32:
            raise ValueError("A.dtype = {} is not float32".format(A.dtype))
        if not A.flags["C_CONTIGUOUS"]:
            raise ValueError("A must be C-contiguous")
        self = cls()
        self.py_buf = {"val": A}
        self.rows, self.cols = A.shape
        self.val = A.ctypes.data_as(POINTER(c_float))
        return self


class ScipyCompressedSparseAllocator(object):
    """Result allocator handed to the C side (pecos/core/base.py:407-478)."""

    CFUNCTYPE = CFUNCTYPE(None, c_bool, c_uint64, c_uint64, c_uint64, c_void_p, c_void_p, c_void_p)

    def __init__(self, rows=0, cols=0, dtype=np.float32):
        assert dtype == np.float32
        self.rows, self.cols = rows, cols
        self.indices = self.indptr = self.data = None
        self.dtype = dtype
        self.is_col_major = None

    def __call__(self, is_col_major, rows, cols, nnz, indices_ptr, indptr_ptr, data_ptr):
        self.rows, self.cols, self.is_col_major = rows, cols, is_col_major
        self.indptr = np.zeros((cols if is_col_major else rows) + 1, dtype=np.uint64)
        self.indices = np.zeros(nnz, dtype=np.uint32)
        self.data = np.zeros(nnz, dtype=self.dtype)
        cast(indices_ptr, POINTER(c_uint64)).contents.value = self.indices.ctypes.data_as(c_void_p).value or 0
        cast(indptr_ptr, POINTER(c_uint64)).contents.value = self.indptr.ctypes.data_as(c_void_p).value or 0
        cast(data_ptr, POINTER(c_uint64)).contents.value = self.data.ctypes.data_as(c_void_p).value or 0

    def get(self):
        # (the reference wraps this with smat_util.csr_matrix, which only widens the index dtype)
        ctor = smat.csc_matrix if self.is_col_major else smat.csr_matrix
        return ctor(
            (self.data, self.indices.astype(np.int64 if self.indices.size >= 2**31 else np.int32),
             self.indptr.astype(np.int64)),
            shape=(self.rows, self.cols),
        )

    @property
    def cfunc(self):
        return self.CFUNCTYPE(self)


class B200CoreLib(object):
    """Loads the CUDA library and declares every reference-compatible symbol (cf. corelib.__init__, base.py:526-539)."""

    def __init__(self, path=LIB_PATH):
        if not os.path.exists(path):
            raise RuntimeError(
                "{} not found: build it first with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(pecos_b200 has no CPU fallback)".format(path)
            )
        self.path = path
        self.clib_float32 = ctypes.CDLL(path)
        self.link_xlinear_methods()
        self.link_ann_hnsw_methods()
        self.link_b200_methods()

    @staticmethod
    def fillprototype(f, restype, argtypes):
        f.restype = restype
        f.argtypes = argtypes

    # ---------------------------------------------------------------- XR-Linear (base.py:799-976)
    def link_xlinear_methods(self):
        c = self.clib_float32
        fp = B200CoreLib.fillprototype
        fp(c.c_xlinear_load_model_from_disk, c_void_p, [c_char_p])
        fp(c.c_xlinear_load_model_from_disk_ext, c_void_p, [c_char_p, c_int])
        fp(c.c_xlinear_load_mmap_model_from_disk, c_void_p, [c_char_p, c_bool])
        fp(c.c_xlinear_compile_mmap_model, None, [c_char_p, c_char_p])
        fp(c.c_xlinear_destruct_model, None, [c_void_p])
        fp(c.c_xlinear_get_int_attr, c_uint32, [c_void_p, c_char_p])
        fp(c.c_xlinear_get_layer_type, c_int, [c_void_p, c_int])
        pred_args = [c_uint32, c_char_p, c_uint32, c_int, ScipyCompressedSparseAllocator.CFUNCTYPE]
        fp(c.c_xlinear_predict_csr_f32, None, [c_void_p, POINTER(ScipyCsrF32)] + pred_args)
        fp(c.c_xlinear_predict_drm_f32, None, [c_void_p, POINTER(ScipyDrmF32)] + pred_args)

        sel_args = [POINTER(ScipyCsrF32), c_char_p, c_int, ScipyCompressedSparseAllocator.CFUNCTYPE]  # pecos/core/base.py:846-876
        fp(c.c_xlinear_predict_on_selected_outputs_csr_f32, None, [c_void_p, POINTER(ScipyCsrF32)] + sel_args)
        fp(c.c_xlinear_predict_on_selected_outputs_drm_f32, None, [c_void_p, POINTER(ScipyDrmF32)] + sel_args)

        # single-layer mmap handles (pecos/core/base.py:541-606)
        fp(c.c_mlmodel_load_mmap_model, c_void_p, [c_char_p, c_bool])
        fp(c.c_mlmodel_destruct_model, None, [c_void_p])
        fp(c.c_mlmodel_get_int_attr, c_uint32, [c_void_p, c_char_p])
        fp(c.c_mlmodel_compile_mmap_model, None, [c_char_p, c_char_p])
        ml_args = [POINTER(ScipyCsrF32), c_char_p, c_uint32, c_int, ScipyCompressedSparseAllocator.CFUNCTYPE]
        fp(c.c_mlmodel_predict_csr_f32, None, [c_void_p, POINTER(ScipyCsrF32)] + ml_args)
        fp(c.c_mlmodel_predict_drm_f32, None, [c_void_p, POINTER(ScipyDrmF32)] + ml_args)
        ml_sel = [POINTER(ScipyCsrF32), POINTER(ScipyCsrF32), c_char_p, c_int, ScipyCompressedSparseAllocator.CFUNCTYPE]
        fp(c.c_mlmodel_predict_on_selected_outputs_csr_f32, None, [c_void_p, POINTER(ScipyCsrF32)] + ml_sel)
        fp(c.c_mlmodel_predict_on_selected_outputs_drm_f32, None, [c_void_p, POINTER(ScipyDrmF32)] + ml_sel)

        single = [POINTER(ScipyCsrF32), POINTER(ScipyCscF32), POINTER(ScipyCscF32), c_char_p, c_uint32, c_int, c_float,
                  ScipyCompressedSparseAllocator.CFUNCTYPE]  # pecos/core/base.py:880-933
        fp(c.c_xlinear_single_layer_predict_csr_f32, None, [POINTER(ScipyCsrF32)] + single)
        fp(c.c_xlinear_single_layer_predict_drm_f32, None, [POINTER(ScipyDrmF32)] + single)
        single_sel = [POINTER(ScipyCsrF32), POINTER(ScipyCsrF32), POINTER(ScipyCscF32), POINTER(ScipyCscF32), c_char_p, c_int, c_float,
                      ScipyCompressedSparseAllocator.CFUNCTYPE]  # pecos/core/base.py:936-976
        fp(c.c_xlinear_single_layer_predict_on_selected_outputs_csr_f32, None, [POINTER(ScipyCsrF32)] + single_sel)
        fp(c.c_xlinear_single_layer_predict_on_selected_outputs_drm_f32, None, [POINTER(ScipyDrmF32)] + single_sel)
        fp(c.pb200_xlinear_host_from_csc, c_void_p, [POINTER(ScipyCscF32), POINTER(ScipyCscF32), c_float])
        fp(c.pb200_layer_cache_clear, c_uint32, [])
        fp(c.pb200_layer_cache_info, None, [POINTER(c_uint64)])

    def xlinear_single_layer_predict(self, X, csr_codes, W, C, post_processor_str, only_topk, num_threads, bias, pred_alloc):
        """Same contract as corelib.xlinear_single_layer_predict (pecos/core/base.py:1160-1226): one layer of the python
        prediction chain.  W / C: csc_matrix (or ScipyCscF32), csr_codes: csr_matrix or None."""
        self.require_gpu()
        clib = self.clib_float32
        if isinstance(X, smat.csr_matrix):
            if not X.has_sorted_indices:
                raise ValueError("Query matrix does not have sorted indices!")
            X = ScipyCsrF32.init_from(X)
        elif isinstance(X, np.ndarray):
            X = ScipyDrmF32.init_from(X)
        if isinstance(X, ScipyCsrF32):
            c_predict = clib.c_xlinear_single_layer_predict_csr_f32
        elif isinstance(X, ScipyDrmF32):
            c_predict = clib.c_xlinear_single_layer_predict_drm_f32
        else:
            raise NotImplementedError("type(X) = {} not implemented".format(type(X)))
        if isinstance(W, smat.csc_matrix):
            W = ScipyCscF32.init_from(W)
        if isinstance(C, smat.csc_matrix):
            C = ScipyCscF32.init_from(C)
        if not isinstance(W, ScipyCscF32) or not isinstance(C, ScipyCscF32):
            raise NotImplementedError("W and C must be csc_matrix / ScipyCscF32")
        if csr_codes is not None and isinstance(csr_codes, smat.csr_matrix):
            csr_codes = ScipyCsrF32.init_from(csr_codes)
        if csr_codes is not None and not isinstance(csr_codes, ScipyCsrF32):
            raise NotImplementedError("type(csr_codes) = {} not implemented".format(type(csr_codes)))
        c_predict(
            byref(X),
            byref(csr_codes) if csr_codes is not None else None,
            byref(W),
            byref(C),
            post_processor_str.encode("utf-8"),
            only_topk,
            num_threads,
            bias,
            pred_alloc.cfunc,
        )

    def xlinear_single_layer_predict_on_selected_outputs(self, X, selected_outputs_csr, csr_codes, W, C, post_processor_str,
                                                         num_threads, bias, pred_alloc):
        """Same contract as corelib.xlinear_single_layer_predict_on_selected_outputs (pecos/core/base.py:1227-1300): one layer,
        scores of exactly the (instance, label) pairs of ``selected_outputs_csr``."""
        self.require_gpu()
        clib = self.clib_float32
        if isinstance(X, smat.csr_matrix):
            if not X.has_sorted_indices:
                raise ValueError("Query matrix does not have sorted indices!")
            X = ScipyCsrF32.init_from(X)
        elif isinstance(X, np.ndarray):
            X = ScipyDrmF32.init_from(X)
        if isinstance(X, ScipyCsrF32):
            c_predict = clib.c_xlinear_single_layer_predict_on_selected_outputs_csr_f32
        elif isinstance(X, ScipyDrmF32):
            c_predict = clib.c_xlinear_single_layer_predict_on_selected_outputs_drm_f32
        else:
            raise NotImplementedError("type(X) = {} not implemented".format(type(X)))
        if isinstance(selected_outputs_csr, smat.csr_matrix):
            selected_outputs_csr = ScipyCsrF32.init_from(selected_outputs_csr.astype(np.float32))
        if not isinstance(selected_outputs_csr, ScipyCsrF32):
            raise NotImplementedError("selected_outputs_csr must be a csr_matrix / ScipyCsrF32")
        if isinstance(W, smat.csc_matrix):
            W = ScipyCscF32.init_from(W)
        if isinstance(C, smat.csc_matrix):
            C = ScipyCscF32.init_from(C)
        if not isinstance(W, ScipyCscF32) or not isinstance(C, ScipyCscF32):
            raise NotImplementedError("W and C must be csc_matrix / ScipyCscF32")
        if csr_codes is not None and isinstance(csr_codes, smat.csr_matrix):
            csr_codes = ScipyCsrF32.init_from(csr_codes)
        if csr_codes is not None and not isinstance(csr_codes, ScipyCsrF32):
            raise NotImplementedError("type(csr_codes) = {} not implemented".format(type(csr_codes)))
        c_predict(
            byref(X),
            byref(selected_outputs_csr),
            byref(csr_codes) if csr_codes is not None else None,
            byref(W),
            byref(C),
            post_processor_str.encode("utf-8"),
            num_threads,
            bias,
            pred_alloc.cfunc,
        )

    def require_gpu(self):
        if self.clib_float32.pb200_device_count() <= 0:
            raise RuntimeError("pecos_b200: no CUDA device visible and there is no CPU fallback")

    def xlinear_load_mmap(self, folder, lazy_load=False):
        self.require_gpu()
        return c_void_p(self.clib_float32.c_xlinear_load_mmap_model_from_disk(folder.encode("utf-8"), c_bool(lazy_load)))

    def xlinear_load_predict_only(self, folder, weight_matrix_type="BINARY_SEARCH_CHUNKED"):
        self.require_gpu()
        type_id = XLINEAR_INFERENCE_MODEL_TYPES[weight_matrix_type]
        return c_void_p(self.clib_float32.c_xlinear_load_model_from_disk_ext(folder.encode("utf-8"), c_int(int(type_id))))

    def xlinear_destruct_model(self, c_model):
        self.clib_float32.c_xlinear_destruct_model(c_model)

    def xlinear_get_int_attr(self, c_model, attr):
        assert attr in {"depth", "nr_features", "nr_labels", "nr_codes"}, f"attr {attr} not implemented"
        return self.clib_float32.c_xlinear_get_int_attr(c_model, attr.encode("utf-8"))

    def xlinear_get_layer_type(self, c_model, layer_depth):
        return self.clib_float32.c_xlinear_get_layer_type(c_model, layer_depth)

    def xlinear_predict(self, c_model, X, overriden_beam_size, overriden_post_processor_str, overriden_only_topk,
                        threads, pred_alloc):
        """Same contract as corelib.xlinear_predict (base.py:1041-1095)."""
        clib = self.clib_float32
        if isinstance(X, smat.csr_matrix):
            if not X.has_sorted_indices:
                raise ValueError("Query matrix does not have sorted indices!")
            X = ScipyCsrF32.init_from(X)
        elif isinstance(X, np.ndarray):
            X = ScipyDrmF32.init_from(X)
        if isinstance(X, ScipyCsrF32):
            c_predict = clib.c_xlinear_predict_csr_f32
        elif isinstance(X, ScipyDrmF32):
            c_predict = clib.c_xlinear_predict_drm_f32
        else:
            raise NotImplementedError("type(X) = {} not implemented".format(type(X)))
        c_predict(
            c_model,
            byref(X),
            overriden_beam_size if overriden_beam_size else 0,
            overriden_post_processor_str.encode("utf-8") if overriden_post_processor_str else None,
            overriden_only_topk if overriden_only_topk else 0,
            threads,
            pred_alloc.cfunc,
        )

    # ---------------------------------------------------------------- HNSW (base.py:1865-1964)
    def xlinear_predict_on_selected_outputs(self, c_model, X, selected_outputs_csr, overriden_post_processor_str, threads, pred_alloc):
        """Argument handling of corelib.xlinear_predict_on_selected_outputs (pecos/core/base.py:1097-1160)."""
        clib = self.clib_float32
        if isinstance(X, smat.csr_matrix):
            if not X.has_sorted_indices:
                raise ValueError("Query matrix does not have sorted indices!")
            X = ScipyCsrF32.init_from(X)
        elif isinstance(X, np.ndarray):
            X = ScipyDrmF32.init_from(X)
        if not isinstance(selected_outputs_csr, smat.csr_matrix):
            raise ValueError("type(selected_outputs_csr) = {} not implemented".format(type(selected_outputs_csr)))
        selected = ScipyCsrF32.init_from(selected_outputs_csr)
        if isinstance(X, ScipyCsrF32):
            c_predict = clib.c_xlinear_predict_on_selected_outputs_csr_f32
        elif isinstance(X, ScipyDrmF32):
            c_predict = clib.c_xlinear_predict_on_selected_outputs_drm_f32
        else:
            raise NotImplementedError("type(X) = {} not implemented".format(type(X)))
        c_predict(
            c_model,
            byref(X),
            byref(selected),
            overriden_post_processor_str.encode("utf-8") if overriden_post_processor_str else None,
            threads,
            pred_alloc.cfunc,
        )

    def link_ann_hnsw_methods(self):
        c = self.clib_float32
        fp = B200CoreLib.fillprototype
        self.ann_hnsw_fn_dict = {}
        for data_type, metric in (("drm", "ip"), ("drm", "l2"), ("csr", "ip"), ("csr", "l2")):
            key = (data_type, metric)
            suffix = "{}_{}_f32".format(data_type, metric)
            mat_t = ScipyDrmF32 if data_type == "drm" else ScipyCsrF32
            if not hasattr(c, "c_ann_hnsw_load_" + suffix):
                continue
            load = getattr(c, "c_ann_hnsw_load_" + suffix)
            fp(load, c_void_p, [c_char_p, c_bool])
            destruct = getattr(c, "c_ann_hnsw_destruct_" + suffix)
            fp(destruct, None, [c_void_p])
            s_create = getattr(c, "c_ann_hnsw_searchers_create_" + suffix)
            fp(s_create, c_void_p, [c_void_p, c_uint32])
            s_destruct = getattr(c, "c_ann_hnsw_searchers_destruct_" + suffix)
            fp(s_destruct, None, [c_void_p])
            predict = getattr(c, "c_ann_hnsw_predict_" + suffix)
            fp(predict, None, [c_void_p, POINTER(mat_t), POINTER(c_uint32), POINTER(c_float), c_uint32,
                               c_uint32, c_int32, c_void_p])
            save = getattr(c, "c_ann_hnsw_save_" + suffix)
            fp(save, None, [c_void_p, c_char_p])
            self.ann_hnsw_fn_dict[key] = {
                "save": save,
                "load": load,
                "destruct": destruct,
                "searchers_create": s_create,
                "searchers_destruct": s_destruct,
                "predict": predict,
            }

    def ann_hnsw_init(self, data_type, metric_type):
        key = (data_type, metric_type)
        if key not in self.ann_hnsw_fn_dict:
            raise NotImplementedError("data_type={}, metric_type={} is not implemented".format(data_type, metric_type))
        return self.ann_hnsw_fn_dict[key]

    # ---------------------------------------------------------------- pb200_* additions
    def link_b200_methods(self):
        c = self.clib_float32
        fp = B200CoreLib.fillprototype
        fp(c.pb200_version, c_char_p, [])
        fp(c.pb200_device_count, c_int, [])
        fp(c.pb200_set_device, c_int, [c_int])
        fp(c.pb200_get_device, c_int, [])
        fp(c.pb200_host_alloc, c_void_p, [c_size_t])
        fp(c.pb200_host_free, None, [c_void_p])
        fp(c.pb200_l2_flush, None, [])
        fp(c.pb200_xlinear_resident_upload_csr, None, [c_void_p, POINTER(ScipyCsrF32)])
        fp(c.pb200_xlinear_resident_predict, c_double, [c_void_p, c_uint32, c_char_p, c_uint32, c_int])
        fp(c.pb200_xlinear_resident_fetch, None, [c_void_p, ScipyCompressedSparseAllocator.CFUNCTYPE])
        fp(c.pb200_xlinear_load_sharded, c_void_p, [c_char_p, c_int, c_uint32, c_uint32])
        fp(c.pb200_xlinear_get_shard, None, [c_void_p, POINTER(c_uint32)])
        fp(c.pb200_xlinear_sharded_local_csr, c_uint32, [c_void_p, POINTER(ScipyCsrF32), c_uint32, c_char_p, c_uint32, c_uint32,
                                                           c_void_p, c_void_p, c_void_p, c_void_p])
        fp(c.pb200_xlinear_sharded_merge, None, [c_void_p, c_uint32, c_uint32, c_uint32, c_uint32, c_void_p, c_void_p, c_void_p,
                                                 c_void_p, ScipyCompressedSparseAllocator.CFUNCTYPE])
        fp(c.pb200_xlinear_sharded_local_csr_packed, c_uint32, [c_void_p, POINTER(ScipyCsrF32), c_uint32, c_char_p, c_uint32, c_uint32,
                                                                  c_void_p])
        fp(c.pb200_xlinear_sharded_merge_packed, None, [c_void_p, c_uint32, c_uint32, c_uint32, c_uint32, c_void_p,
                                                        ScipyCompressedSparseAllocator.CFUNCTYPE])
        fp(c.pb200_xlinear_set_profile, None, [c_void_p, c_int])
        fp(c.pb200_xlinear_reset_profile, None, [c_void_p])
        fp(c.pb200_xlinear_set_lookup, c_int, [c_void_p, c_int])
        fp(c.pb200_xlinear_get_profile, None, [c_void_p, POINTER(c_double)])
        fp(c.pb200_xlinear_get_kernel_ids, None, [c_void_p, POINTER(c_int)])
        fp(c.pb200_xlinear_get_stats, None, [c_void_p, POINTER(c_uint64)])
        fp(c.pb200_xlinear_launches, c_uint64, [c_void_p])
        fp(c.pb200_xlinear_model_bytes, c_uint64, [c_void_p])
        fp(c.pb200_xlinear_replicas, c_uint32, [c_void_p])
        fp(c.pb200_hnsw_replicas, c_uint32, [c_void_p])
        fp(c.pb200_hnsw_vcap_retries, c_uint32, [c_void_p])
        fp(c.pb200_hnsw_resident_upload, None, [c_void_p, POINTER(ScipyDrmF32)])
        fp(c.pb200_hnsw_resident_upload_csr, None, [c_void_p, POINTER(ScipyCsrF32)])
        fp(c.pb200_hnsw_sparse_entries, c_uint64, [c_void_p])
        fp(c.pb200_hnsw_resident_predict, c_double, [c_void_p, c_uint32, c_uint32])
        fp(c.pb200_hnsw_resident_fetch, None, [c_void_p, POINTER(c_uint32), POINTER(c_float)])
        fp(c.pb200_hnsw_get_counters, None, [c_void_p, POINTER(c_uint64)])
        fp(c.pb200_hnsw_set_stages, c_int, [c_void_p, c_int])
        fp(c.pb200_hnsw_get_info, None, [c_void_p, POINTER(c_uint64)])
        fp(c.pb200_hnsw_host_info, c_int, [c_char_p, c_int, c_int, POINTER(c_uint64)])
        fp(c.pb200_hnsw_build_sparse_knn, c_int, [c_int, c_void_p, c_uint32, c_uint32, c_int] + [c_void_p] * 8)
        fp(c.pb200_hnsw_build_sparse_select, c_int, [c_int, c_void_p, c_uint32, c_uint32, c_uint32, c_int] + [c_void_p] * 6)
        fp(c.pb200_xlinear_host_load, c_void_p, [c_char_p, c_int])
        fp(c.pb200_xlinear_host_free, None, [c_void_p])
        fp(c.pb200_xlinear_host_depth, c_uint32, [c_void_p])
        fp(c.pb200_xlinear_host_layer_dims, None, [c_void_p, c_uint32, POINTER(c_uint64)])
        fp(c.pb200_xlinear_host_layer_export, None, [c_void_p, c_uint32, c_void_p, c_void_p, c_void_p, c_void_p])

    def device_count(self):
        return int(self.clib_float32.pb200_device_count())

    def set_device(self, device):
        if self.clib_float32.pb200_set_device(int(device)) != 0:
            raise RuntimeError("pecos_b200: cannot select CUDA device {}".format(device))

    def pinned_empty(self, n, dtype):
        """numpy array backed by cudaMallocHost memory (freed when the array's base object is collected)."""
        dtype = np.dtype(dtype)
        nbytes = max(1, int(n) * dtype.itemsize)
        ptr = self.clib_float32.pb200_host_alloc(nbytes)
        if not ptr:
            raise MemoryError("pb200_host_alloc failed")
        buf = (ctypes.c_char * nbytes).from_address(ptr)
        owner = _PinnedOwner(self, ptr, buf)
        arr = np.frombuffer(owner.buf, dtype=dtype, count=int(n))
        return _PinnedArray(arr, owner)

    def host_layer_layout_from_csc(self, W, C, bias):
        """Host-only: the chunk layout the single-layer entry point builds from in-memory W / C (csc_matrix)."""
        cw = ScipyCscF32.init_from(smat.csc_matrix(W, dtype=np.float32))
        cc = ScipyCscF32.init_from(smat.csc_matrix(C, dtype=np.float32))
        h = c_void_p(self.clib_float32.pb200_xlinear_host_from_csc(byref(cw), byref(cc), c_float(bias)))
        return self._export_host_model(h)

    def host_model_layout(self, model_path, is_mmap=False):
        """Host-only: load a model folder and return its chunk layout per layer as numpy arrays (no GPU needed)."""
        c = self.clib_float32
        h = c_void_p(c.pb200_xlinear_host_load(model_path.encode("utf-8"), 1 if is_mmap else 0))
        return self._export_host_model(h)

    def _export_host_model(self, h):
        c = self.clib_float32
        try:
            layers = []
            for d in range(c.pb200_xlinear_host_depth(h)):
                dims = (c_uint64 * 8)()
                c.pb200_xlinear_host_layer_dims(h, d, dims)
                w_rows, n_cols, out_cols, n_chunks, c_max, meta_len, n_ent, n_lab = [int(x) for x in dims]
                chunks = np.zeros(n_chunks, dtype=CHUNK_HEADER_DTYPE)
                meta = np.zeros(meta_len, dtype=np.uint32)
                entries = np.zeros(n_ent, dtype=CHUNK_ENTRY_DTYPE)
                lab = np.zeros(n_lab, dtype=np.uint32)
                c.pb200_xlinear_host_layer_export(h, d, chunks.ctypes.data_as(c_void_p), meta.ctypes.data_as(c_void_p),
                                                  entries.ctypes.data_as(c_void_p), lab.ctypes.data_as(c_void_p))
                layers.append(dict(w_rows=w_rows, n_cols=n_cols, out_cols=out_cols, n_chunks=n_chunks, c_max=c_max,
                                   chunks=chunks, meta=meta, entries=entries, label_of_col=lab))
            return layers
        finally:
            c.pb200_xlinear_host_free(h)


CHUNK_HEADER_DTYPE = np.dtype(
    [("col_begin", "<u4"), ("n_cols", "<u4"), ("nnz_rows", "<u4"), ("has_bias", "<u4"), ("meta_off", "<u8"), ("ent_off", "<u8")]
)
CHUNK_ENTRY_DTYPE = np.dtype([("col_offset", "<u4"), ("val", "<f4")])

class _PinnedOwner(object):
    def __init__(self, lib, ptr, buf):
        self.lib, self.ptr, self.buf = lib, ptr, buf

    def __del__(self):
        try:
            self.lib.clib_float32.pb200_host_free(c_void_p(self.ptr))
        except Exception:
            pass


class _PinnedArray(object):
    """Tiny holder keeping the pinned allocation alive next to the numpy view onto it."""

    def __init__(self, array, owner):
        self.array = array
        self._owner = owner


_clib = None


def get_clib():
    """Process-wide singleton, like ``pecos.core.clib`` (base.py:2429)."""
    global _clib
    if _clib is None:
        _clib = B200CoreLib()
    return _clib
