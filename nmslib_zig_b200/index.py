"""Host-side mirror of lib.zig's `Index` over the C ABI of libnmslib_b200.so.

Zig is not available in this image, so the host layer that lib.zig provides
(lib.zig:495-1270) is mirrored here 1:1 in Python over ctypes: same method names
(camelCase kept on purpose), same argument meaning, same error mapping
(lib.zig:29-74), and -- the one deliberate difference, SURVEY Appendix E --
`knnQueryBatch` issues ONE `nmslib_knn_query_batch` call for the whole batch instead
of a per-query loop (lib.zig:905-928).  Nothing in here computes distances: every
query goes through the C ABI into the CUDA engine, and the import fails loudly if the
shared library is missing.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path
from typing import Optional, Sequence

import numpy as np

_PKG = Path(__file__).resolve().parent
# NB200_LIB: the tools point this at lib/libnmslib_b200_exp.so (the -DNB200_EXPERIMENTS build with the timing knobs)
LIB_PATH = Path(os.environ["NB200_LIB"]) if os.environ.get("NB200_LIB") else _PKG / "lib" / "libnmslib_b200.so"

# ---- nmslib_b200.h types -------------------------------------------------------------
DATATYPE = {"DenseVector": 0, "SparseVector": 1, "DenseUInt8Vector": 2, "ObjectAsString": 3}
DISTTYPE = {"Float": 0, "Int": 1}


class NmslibError(RuntimeError):
    """lib.zig:11-27 / :29-74 -- one error name per nmslib_error_t code."""

    NAMES = {
        1: "NullPointer", 2: "InvalidArgument", 3: "OutOfMemory", 4: "BufferTooSmall",
        5: "SpaceIncompatible", 6: "QueryTooLarge", 7: "InvalidSparseElement", 8: "IndexBuildFailed",
        9: "QueryExecutionFailed", 10: "DataIOFailed", 11: "PluginRegistrationFailed", 12: "Internal",
        13: "Runtime", 14: "IndexNotBuilt",
    }

    def __init__(self, code: int, message: str = ""):
        self.code = code
        self.name = self.NAMES.get(code, f"Unknown({code})")
        super().__init__(f"error.{self.name}: {message}")


class Result(C.Structure):
    _fields_ = [("ids", C.POINTER(C.c_int32)), ("distances", C.POINTER(C.c_float)),
                ("size", C.c_size_t), ("capacity", C.c_size_t)]


_ALLOC_FN = C.CFUNCTYPE(C.c_void_p, C.c_size_t, C.c_void_p)
_FREE_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p)


class Allocator(C.Structure):
    _fields_ = [("alloc", _ALLOC_FN), ("free", _FREE_FN), ("ctx", C.c_void_p)]


class ErrorDetail(C.Structure):
    _fields_ = [("code", C.c_int), ("message", C.c_void_p), ("file", C.c_void_p), ("line", C.c_int)]


class Stats(C.Structure):
    _fields_ = [("queries", C.c_uint64), ("kernel_launches", C.c_uint64), ("distance_evals", C.c_uint64),
                ("hnsw_expansions", C.c_uint64), ("last_kernel_ms", C.c_double), ("last_total_ms", C.c_double),
                ("fallback_queries", C.c_uint64), ("device_bytes", C.c_uint64), ("last_scan_ms", C.c_double),
                ("scan_ms_sum", C.c_double), ("scan_count", C.c_uint64), ("build_total_ms", C.c_double),
                ("build_scan_ms", C.c_double), ("build_select_ms", C.c_double), ("build_link_ms", C.c_double),
                ("build_batches", C.c_uint64), ("build_prunes", C.c_uint64), ("split_queries", C.c_uint64),
                ("u8_imma", C.c_uint64), ("uploaded_rows", C.c_uint64), ("range_tc_queries", C.c_uint64),
                ("range_fallback_queries", C.c_uint64)]


# every symbol include/nmslib_b200.h declares (the CPU-side test checks this list against the header)
ABI_SYMBOLS = [
    "nmslib_init", "nmslib_index_create", "nmslib_index_destroy", "nmslib_create_index", "nmslib_reset_index",
    "nmslib_create_params", "nmslib_add_param", "nmslib_free_params", "nmslib_get_space_type", "nmslib_get_method",
    "nmslib_free_string", "nmslib_get_last_error_detail", "nmslib_add_data_point", "nmslib_add_data_point_batch",
    "nmslib_add_data_point_batch_uint8", "nmslib_add_data_point_batch_string",
    "nmslib_add_data_point_batch_pointers", "nmslib_knn_query_get_size", "nmslib_knn_query_fill",
    "nmslib_knn_query_batch", "nmslib_range_query_get_size", "nmslib_range_query_fill", "nmslib_get_distance",
    "nmslib_get_data_point_size", "nmslib_get_data_point_fill", "nmslib_get_data_point_string",
    "nmslib_borrow_data_dense", "nmslib_borrow_data_sparse", "nmslib_save_index", "nmslib_load_index",
    "nmslib_set_query_time_params", "nmslib_set_thread_pool_size", "nmslib_get_thread_pool_size", "nmslib_data_qty",
    "nmslib_index_memory_usage", "nmslib_initialize_pool", "nmslib_free_result",
]
EXT_SYMBOLS = [
    "nmslib_b200_set_device", "nmslib_b200_device_available", "nmslib_b200_set_shard", "nmslib_b200_import_hnsw",
    "nmslib_b200_prepare", "nmslib_b200_knn_device", "nmslib_b200_merge_topk", "nmslib_b200_get_stats",
    "nmslib_b200_version", "nmslib_b200_scan_plan", "nmslib_b200_scan_plan_pairs", "nmslib_b200_set_option",
    "nmslib_b200_shard_export", "nmslib_b200_shard_connect", "nmslib_b200_shard_disconnect",
    "nmslib_b200_range_query_batch",
]

_lib = None
_libc = C.CDLL(None)
_libc.malloc.restype = C.c_void_p
_libc.malloc.argtypes = [C.c_size_t]
_libc.free.argtypes = [C.c_void_p]
_live_allocs = 0


def _alloc_cb(size, _ctx):
    global _live_allocs
    _live_allocs += 1
    return _libc.malloc(size)


def _free_cb(ptr, _ctx):
    global _live_allocs
    if ptr:
        _live_allocs -= 1
        _libc.free(ptr)


# keep the callback objects alive for the life of the process
_ALLOC = Allocator(_ALLOC_FN(_alloc_cb), _FREE_FN(_free_cb), None)


def live_allocations() -> int:
    """std.testing.allocator stand-in: allocations made through the callbacks and not yet freed."""
    return _live_allocs


def lib() -> C.CDLL:
    """Load libnmslib_b200.so (fails loudly when it has not been built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(f"{LIB_PATH} is missing: run `python -m nmslib_zig_b200.build` (no CPU fallback exists)")
    L = C.CDLL(str(LIB_PATH))
    vp, sz, i32p, f32p = C.c_void_p, C.c_size_t, C.POINTER(C.c_int32), C.POINTER(C.c_float)
    ap = C.POINTER(Allocator)
    sig = {
        "nmslib_init": (None, []),
        "nmslib_index_create": (C.c_int, [C.c_char_p, vp, C.c_char_p, C.c_int, C.c_int, ap, C.POINTER(vp)]),
        "nmslib_index_destroy": (None, [vp]),
        "nmslib_create_index": (C.c_int, [vp, vp, C.c_int]),
        "nmslib_reset_index": (C.c_int, [vp]),
        "nmslib_create_params": (vp, [ap]),
        "nmslib_add_param": (C.c_int, [vp, C.c_char_p, C.c_int, vp]),
        "nmslib_free_params": (None, [vp]),
        "nmslib_get_space_type": (C.c_int, [vp, C.POINTER(vp), C.POINTER(sz), ap]),
        "nmslib_get_method": (C.c_int, [vp, C.POINTER(vp), C.POINTER(sz), ap]),
        "nmslib_free_string": (None, [vp, ap]),
        "nmslib_get_last_error_detail": (C.c_int, [C.POINTER(ErrorDetail), ap]),
        "nmslib_add_data_point": (C.c_int, [vp, vp, sz, C.c_int32]),
        "nmslib_add_data_point_batch": (C.c_int, [vp, vp, sz, sz, i32p, C.POINTER(sz)]),
        "nmslib_add_data_point_batch_uint8": (C.c_int, [vp, vp, sz, sz, i32p]),
        "nmslib_add_data_point_batch_string": (C.c_int, [vp, C.POINTER(C.c_char_p), sz, i32p]),
        "nmslib_add_data_point_batch_pointers": (C.c_int, [vp, C.c_int, C.POINTER(vp), sz, sz, i32p, C.POINTER(sz)]),
        "nmslib_knn_query_get_size": (C.c_int, [vp, vp, sz, sz, C.POINTER(sz), sz]),
        "nmslib_knn_query_fill": (C.c_int, [vp, vp, sz, sz, C.POINTER(Result), sz]),
        "nmslib_knn_query_batch": (C.c_int, [vp, vp, sz, sz, sz, C.POINTER(Result), C.POINTER(sz), sz]),
        "nmslib_range_query_get_size": (C.c_int, [vp, vp, sz, C.c_double, C.POINTER(sz), sz]),
        "nmslib_range_query_fill": (C.c_int, [vp, vp, sz, C.c_double, C.POINTER(Result), sz]),
        "nmslib_get_distance": (C.c_int, [vp, sz, sz, f32p]),
        "nmslib_get_data_point_size": (C.c_int, [vp, sz, C.POINTER(sz)]),
        "nmslib_get_data_point_fill": (C.c_int, [vp, sz, vp, sz]),
        "nmslib_get_data_point_string": (C.c_int, [vp, sz, C.POINTER(vp), C.POINTER(sz), ap]),
        "nmslib_borrow_data_dense": (C.c_int, [vp, sz, C.POINTER(vp), C.POINTER(sz), C.POINTER(vp)]),
        "nmslib_borrow_data_sparse": (C.c_int, [vp, sz, C.POINTER(vp), C.POINTER(sz), C.POINTER(vp)]),
        "nmslib_save_index": (C.c_int, [vp, C.c_char_p, C.c_int]),
        "nmslib_load_index": (C.c_int, [C.c_char_p, C.c_int, C.c_int, ap, C.c_int, C.POINTER(vp)]),
        "nmslib_set_query_time_params": (C.c_int, [vp, vp]),
        "nmslib_set_thread_pool_size": (C.c_int, [vp, sz]),
        "nmslib_get_thread_pool_size": (sz, [vp]),
        "nmslib_data_qty": (sz, [vp]),
        "nmslib_index_memory_usage": (sz, [vp]),
        "nmslib_initialize_pool": (None, [vp]),
        "nmslib_free_result": (None, [C.POINTER(Result)]),
        "nmslib_b200_set_device": (C.c_int, [C.c_int]),
        "nmslib_b200_device_available": (C.c_int, []),
        "nmslib_b200_set_shard": (C.c_int, [vp, C.c_uint32]),
        "nmslib_b200_import_hnsw": (C.c_int, [vp, C.c_char_p]),
        "nmslib_b200_prepare": (C.c_int, [vp]),
        "nmslib_b200_knn_device": (C.c_int, [vp, vp, sz, sz, sz, vp, vp, vp, vp]),
        "nmslib_b200_merge_topk": (C.c_int, [vp, vp, vp, sz, sz, sz, vp, vp, vp]),
        "nmslib_b200_get_stats": (C.c_int, [vp, C.POINTER(Stats)]),
        "nmslib_b200_version": (C.c_char_p, []),
        "nmslib_b200_set_option": (C.c_int, [C.c_char_p, C.c_int]),
        "nmslib_b200_shard_export": (C.c_int, [vp, sz, sz, vp]),
        "nmslib_b200_shard_connect": (C.c_int, [vp, C.c_int, C.c_int, vp]),
        "nmslib_b200_shard_disconnect": (C.c_int, [vp]),
        "nmslib_b200_range_query_batch": (C.c_int, [vp, vp, sz, sz, C.POINTER(C.c_double), C.POINTER(Result)]),
        "nmslib_b200_scan_plan": (sz, [sz, sz, sz, C.c_int, vp, sz, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
        "nmslib_b200_scan_plan_pairs": (sz, [sz, sz, sz, C.c_int, vp, sz, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)  # AttributeError here == a symbol the header promises is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def last_error_message() -> str:
    L = lib()
    d = ErrorDetail()
    if L.nmslib_get_last_error_detail(C.byref(d), C.byref(_ALLOC)) != 0:
        return ""
    msg = C.string_at(d.message).decode(errors="replace") if d.message else ""
    L.nmslib_free_string(d.message, C.byref(_ALLOC))
    L.nmslib_free_string(d.file, C.byref(_ALLOC))
    return msg


def _check(rc: int):
    if rc != 0:
        raise NmslibError(rc, last_error_message())


class Params:
    """lib.zig:260-348"""

    def __init__(self, pairs: Optional[dict] = None):
        self.handle = lib().nmslib_create_params(C.byref(_ALLOC))
        if not self.handle:
            raise NmslibError(3, "params")
        for k, v in (pairs or {}).items():
            self.add(k, v)

    def add(self, key: str, value):
        L = lib()
        if isinstance(value, bool):
            value = int(value)
        if isinstance(value, int):
            v = C.c_int(value)
            rc = L.nmslib_add_param(self.handle, key.encode(), 0, C.byref(v))
        elif isinstance(value, float):
            v = C.c_double(value)
            rc = L.nmslib_add_param(self.handle, key.encode(), 1, C.byref(v))
        else:
            v = C.create_string_buffer(str(value).encode())
            rc = L.nmslib_add_param(self.handle, key.encode(), 2, v)
        _check(rc)

    def deinit(self):
        if self.handle:
            lib().nmslib_free_params(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.deinit()
        except Exception:
            pass


class QueryResult:
    """lib.zig:380-401"""

    def __init__(self, ids: np.ndarray, distances: np.ndarray):
        self.ids = ids
        self.distances = distances


class BatchResult:
    """lib.zig:403-412 -- here two [Q, k] slabs plus the per-query found count."""

    def __init__(self, ids: np.ndarray, distances: np.ndarray, sizes: np.ndarray):
        self.ids, self.distances, self.sizes = ids, distances, sizes

    @property
    def results(self):
        return [QueryResult(self.ids[i, : self.sizes[i]], self.distances[i, : self.sizes[i]])
                for i in range(len(self.sizes))]


class Index:
    """lib.zig:495-1270 (dense-vector subset; sparse / string calls raise error.SpaceIncompatible)."""

    def __init__(self, space_type: str, index_params: Optional[Params], method: str,
                 data_type: str = "DenseVector", dist_type: str = "Float", _handle=None):
        L = lib()
        L.nmslib_init()
        self.data_type, self.dist_type = data_type, dist_type
        self.built = False
        if _handle is not None:
            self.handle = _handle
            self.built = True
            return
        effective = "cosinesimil" if space_type == "cosine" else space_type  # lib.zig:530-533
        h = C.c_void_p()
        rc = L.nmslib_index_create(effective.encode(), index_params.handle if index_params else None,
                                   method.encode(), DATATYPE[data_type], DISTTYPE[dist_type], C.byref(_ALLOC),
                                   C.byref(h))
        _check(rc)
        self.handle = h

    # lib.zig spells it `init`; keep an alias so ported tests read the same
    @classmethod
    def init(cls, space_type, index_params, method, data_type="DenseVector", dist_type="Float"):
        return cls(space_type, index_params, method, data_type, dist_type)

    def deinit(self):
        if getattr(self, "handle", None):
            lib().nmslib_index_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.deinit()
        except Exception:
            pass

    def reset(self):
        _check(lib().nmslib_reset_index(self.handle))
        self.built = False

    # -- ingest ------------------------------------------------------------------------
    def addDenseBatch(self, data, ids: Optional[Sequence[int]] = None):
        """lib.zig:702-722.  `data` is [n, dim] float32 (lib.zig substitutes the row position for id 0, :655)."""
        a = np.ascontiguousarray(data, np.float32)
        ids_a = None if ids is None else np.ascontiguousarray(ids, np.int32)
        _check(lib().nmslib_add_data_point_batch(
            self.handle, a.ctypes.data, a.shape[0], a.shape[1],
            None if ids_a is None else ids_a.ctypes.data_as(C.POINTER(C.c_int32)), None))

    def addUInt8Batch(self, data, ids: Optional[Sequence[int]] = None):
        """lib.zig:757-777"""
        a = np.ascontiguousarray(data, np.uint8)
        ids_a = None if ids is None else np.ascontiguousarray(ids, np.int32)
        _check(lib().nmslib_add_data_point_batch_uint8(
            self.handle, a.ctypes.data, a.shape[0], a.shape[1],
            None if ids_a is None else ids_a.ctypes.data_as(C.POINTER(C.c_int32))))

    def addSparseBatch(self, data, ids=None):
        raise NmslibError(5, "sparse vectors stay on the reference CPU code")

    def addStringBatch(self, data, ids=None):
        arr = (C.c_char_p * len(data))(*[d.encode() if isinstance(d, str) else d for d in data])
        _check(lib().nmslib_add_data_point_batch_string(self.handle, arr, len(data), None))

    def buildIndex(self, index_params: Optional[Params] = None, print_progress: bool = False):
        """lib.zig:625-681"""
        _check(lib().nmslib_create_index(self.handle, index_params.handle if index_params else None,
                                         int(print_progress)))
        self.built = True

    def importHnsw(self, path: str):
        """nmslib_b200 extension: adopt a graph written by the reference's Hnsw::SaveIndex."""
        _check(lib().nmslib_b200_import_hnsw(self.handle, str(path).encode()))
        self.built = True

    # -- queries -----------------------------------------------------------------------
    def _elem_dtype(self):
        return np.uint8 if self.data_type == "DenseUInt8Vector" else np.float32

    def knnQuery(self, query, k: int) -> QueryResult:
        """lib.zig:799-887: get_size + fill for ONE query (a batch of one on the device)."""
        L = lib()
        if not self.built:
            self.buildIndex(None, False)
        L.nmslib_initialize_pool(self.handle)
        q = np.ascontiguousarray(query, self._elem_dtype()).reshape(-1)
        need = C.c_size_t()
        _check(L.nmslib_knn_query_get_size(self.handle, q.ctypes.data, q.size, k, C.byref(need), 0))
        ids = np.empty(need.value, np.int32)
        dists = np.empty(need.value, np.float32)
        res = Result(ids.ctypes.data_as(C.POINTER(C.c_int32)), dists.ctypes.data_as(C.POINTER(C.c_float)), 0,
                     need.value)
        _check(L.nmslib_knn_query_fill(self.handle, q.ctypes.data, q.size, k, C.byref(res), 0))
        return QueryResult(ids[: res.size], dists[: res.size])

    def knnQueryBatch(self, queries, k: int, thread_pool_size: Optional[int] = None) -> BatchResult:
        """lib.zig:889-931, re-shaped per SURVEY Appendix E: one flat buffer, two result slabs,
        ONE nmslib_knn_query_batch call."""
        L = lib()
        if not self.built:
            self.buildIndex(None, False)
        L.nmslib_initialize_pool(self.handle)
        q = np.ascontiguousarray(queries, self._elem_dtype())
        if q.ndim != 2:
            raise NmslibError(2, "queries must be [Q, dim]")
        nq, dim = q.shape
        if nq == 0:
            return BatchResult(np.empty((0, k), np.int32), np.empty((0, k), np.float32), np.empty(0, np.int64))
        ids = np.empty((nq, k), np.int32)
        dists = np.empty((nq, k), np.float32)
        # the descriptor table of a batch shape is kept between calls (taken out while in use: a concurrent caller
        # builds its own) and filled without a Python-level loop over ctypes objects
        cached, self._batch_tbl = getattr(self, "_batch_tbl", None), None
        if cached is None or cached[0] != (nq, k):
            results = (Result * nq)()
            tbl = np.frombuffer(results, dtype=np.uint64).reshape(nq, 4)
            tbl[:, 3] = k
            cached = ((nq, k), results, tbl, np.arange(nq, dtype=np.uint64) * np.uint64(4 * k))
        _, results, tbl, off = cached
        tbl[:, 0] = off + np.uint64(ids.ctypes.data)
        tbl[:, 1] = off + np.uint64(dists.ctypes.data)
        tbl[:, 2] = 0
        _check(L.nmslib_knn_query_batch(self.handle, q.ctypes.data, nq, dim, k, results, None,
                                        thread_pool_size or 0))
        sizes = tbl[:, 2].astype(np.int64)
        self._batch_tbl = cached
        if sizes.min() < k:                        # rows with fewer than k answers: id -1 / distance +inf behind them
            short = np.arange(k)[None, :] >= sizes[:, None]
            ids[short] = -1
            dists[short] = np.inf
        return BatchResult(ids, dists, sizes)

    def rangeQuery(self, query, radius: float, capacity: Optional[int] = None):
        """lib.zig:933-974: size estimate (128, nmslib_c.cpp:1046), then fill.  Objects within the radius come
        back in position order, truncated to the buffer (`capacity` overrides the estimate)."""
        L = lib()
        if not self.built:
            self.buildIndex(None, False)
        q = np.ascontiguousarray(query, self._elem_dtype()).reshape(-1)
        need = C.c_size_t()
        _check(L.nmslib_range_query_get_size(self.handle, q.ctypes.data, q.size, radius, C.byref(need), 0))
        cap = int(capacity) if capacity else need.value
        ids = np.empty(cap, np.int32)
        dists = np.empty(cap, np.float32)
        res = Result(ids.ctypes.data_as(C.POINTER(C.c_int32)), dists.ctypes.data_as(C.POINTER(C.c_float)), 0, cap)
        _check(L.nmslib_range_query_fill(self.handle, q.ctypes.data, q.size, radius, C.byref(res), 0))
        return QueryResult(ids[: res.size], dists[: res.size])

    def rangeQueryBatch(self, queries, radius, capacity=128) -> BatchResult:
        """nmslib_b200 extension: ONE nmslib_b200_range_query_batch call for [Q, dim] queries.  `radius` and
        `capacity` are scalars or [Q] arrays.  Every row is what rangeQuery returns for that query (objects within
        the radius in position order, truncated to the capacity), padded to the largest capacity with id -1 /
        distance +inf; `sizes` holds the counts."""
        L = lib()
        if not self.built:
            self.buildIndex(None, False)
        q = np.ascontiguousarray(queries, self._elem_dtype())
        if q.ndim != 2:
            raise NmslibError(2, "queries must be [Q, dim]")
        nq, dim = q.shape
        radii = np.ascontiguousarray(np.broadcast_to(np.asarray(radius, np.float64), (nq,)))
        caps = np.broadcast_to(np.asarray(capacity, np.int64), (nq,))
        if nq and caps.min() < 0:
            raise NmslibError(2, "negative capacity")
        width = int(caps.max()) if nq else 0
        ids = np.full((nq, width), -1, np.int32)
        dists = np.full((nq, width), np.inf, np.float32)
        if nq == 0:
            return BatchResult(ids, dists, np.empty(0, np.int64))
        results = (Result * nq)()
        tbl = np.frombuffer(results, dtype=np.uint64).reshape(nq, 4)
        row = np.arange(nq, dtype=np.uint64) * np.uint64(4 * width)
        tbl[:, 0] = row + np.uint64(ids.ctypes.data)
        tbl[:, 1] = row + np.uint64(dists.ctypes.data)
        tbl[:, 2] = 0
        tbl[:, 3] = caps.astype(np.uint64)
        _check(L.nmslib_b200_range_query_batch(self.handle, q.ctypes.data, nq, dim,
                                               radii.ctypes.data_as(C.POINTER(C.c_double)), results))
        sizes = tbl[:, 2].astype(np.int64)
        return BatchResult(ids, dists, sizes)

    # -- data access ---------------------------------------------------------------------
    def getDistance(self, pos1: int, pos2: int) -> float:
        d = C.c_float()
        _check(lib().nmslib_get_distance(self.handle, pos1, pos2, C.byref(d)))
        return d.value

    def getDataPoint(self, pos: int) -> np.ndarray:
        n = C.c_size_t()
        _check(lib().nmslib_get_data_point_size(self.handle, pos, C.byref(n)))
        out = np.empty(n.value, self._elem_dtype())
        _check(lib().nmslib_get_data_point_fill(self.handle, pos, out.ctypes.data, n.value))
        return out

    def borrowDataDense(self, pos: int) -> np.ndarray:
        data, n, fn = C.c_void_p(), C.c_size_t(), C.c_void_p()
        _check(lib().nmslib_borrow_data_dense(self.handle, pos, C.byref(data), C.byref(n), C.byref(fn)))
        out = np.ctypeslib.as_array(C.cast(data, C.POINTER(C.c_float)), shape=(n.value // 4,)).copy()
        C.CFUNCTYPE(None, C.c_void_p)(fn.value)(data)
        return out

    # -- persistence ---------------------------------------------------------------------
    def save(self, path: str, save_data: bool = True):
        _check(lib().nmslib_save_index(self.handle, str(path).encode(), int(save_data)))

    @classmethod
    def load(cls, path: str, data_type: str = "DenseVector", dist_type: str = "Float", load_data: bool = True):
        h = C.c_void_p()
        _check(lib().nmslib_load_index(str(path).encode(), DATATYPE[data_type], DISTTYPE[dist_type],
                                       C.byref(_ALLOC), int(load_data), C.byref(h)))
        return cls("", None, "", data_type, dist_type, _handle=h)

    # -- settings / introspection ----------------------------------------------------------
    def setQueryTimeParams(self, params: Params):
        _check(lib().nmslib_set_query_time_params(self.handle, params.handle))

    def setThreadPoolSize(self, size: int):
        _check(lib().nmslib_set_thread_pool_size(self.handle, size))

    def getThreadPoolSize(self) -> int:
        return lib().nmslib_get_thread_pool_size(self.handle)

    def dataQty(self) -> int:
        return lib().nmslib_data_qty(self.handle)

    def _get_str(self, fn) -> str:
        s, n = C.c_void_p(), C.c_size_t()
        _check(fn(self.handle, C.byref(s), C.byref(n), C.byref(_ALLOC)))
        out = C.string_at(s, n.value).decode()
        lib().nmslib_free_string(s, C.byref(_ALLOC))
        return out

    def getSpaceType(self) -> str:
        return self._get_str(lib().nmslib_get_space_type)

    def getMethod(self) -> str:
        return self._get_str(lib().nmslib_get_method)

    def getDataType(self) -> str:
        return self.data_type

    def memoryUsage(self) -> int:
        return lib().nmslib_index_memory_usage(self.handle)

    # -- nmslib_b200 extensions --------------------------------------------------------------
    def setShard(self, pos_base: int):
        _check(lib().nmslib_b200_set_shard(self.handle, pos_base))

    def prepare(self):
        _check(lib().nmslib_b200_prepare(self.handle))

    def stats(self) -> dict:
        s = Stats()
        _check(lib().nmslib_b200_get_stats(self.handle, C.byref(s)))
        return {f: getattr(s, f) for f, _ in Stats._fields_}

    def knnDevice(self, d_queries_ptr: int, nq: int, dim: int, k: int, d_ids_ptr: int, d_dists_ptr: int,
                  d_keys_ptr: int = 0, stream: int = 0):
        """Device-resident query: raw device pointers (e.g. torch.Tensor.data_ptr()); the queries are float32, or
        uint8 for a DenseUInt8Vector index (seq_search or hnsw)."""
        _check(lib().nmslib_b200_knn_device(self.handle, d_queries_ptr, nq, dim, k, d_ids_ptr, d_dists_ptr,
                                            d_keys_ptr or None, stream or None))

    # -- row shards across processes (one rank per GPU): include/nmslib_b200.h, mode (B) --------------------
    def shardExport(self, max_queries: int, max_k: int) -> bytes:
        """This rank's exchange window; returns the 256-byte blob the launcher all-gathers."""
        blob = C.create_string_buffer(256)
        _check(lib().nmslib_b200_shard_export(self.handle, max_queries, max_k, blob))
        return blob.raw

    def shardConnect(self, rank: int, world: int, blobs: bytes):
        """blobs = the ranks' blobs concatenated in rank order; afterwards every knn call returns the global top-k."""
        assert len(blobs) == 256 * world
        buf = C.create_string_buffer(bytes(blobs), len(blobs))
        _check(lib().nmslib_b200_shard_connect(self.handle, rank, world, buf))

    def shardDisconnect(self):
        _check(lib().nmslib_b200_shard_disconnect(self.handle))

    def mergeTopk(self, d_keys_ptr: int, d_ids_ptr: int, lists: int, nq: int, k: int, d_out_ids_ptr: int,
                  d_out_dists_ptr: int, stream: int = 0):
        """d_ids_ptr = 0: the external ids are the global positions in the keys (no id lists to exchange)."""
        _check(lib().nmslib_b200_merge_topk(self.handle, d_keys_ptr, d_ids_ptr or None, lists, nq, k, d_out_ids_ptr,
                                            d_out_dists_ptr, stream or None))


def device_available() -> bool:
    return bool(lib().nmslib_b200_device_available())


def set_device(device: int):
    lib().nmslib_b200_set_device(device)


def scan_plan(nq: int, n: int, k: int, sm_count: int = 148):
    """Work decomposition of the tensor-core scan (host logic only): (pieces[m,5], n_cta, s_max) with
    pieces = {cta, query block, first tile, end tile, slot}."""
    L = lib()
    nc, sm = C.c_int(0), C.c_int(0)
    m = L.nmslib_b200_scan_plan(nq, n, k, sm_count, None, 0, C.byref(nc), C.byref(sm))
    out = np.zeros((m, 5), np.int32)
    L.nmslib_b200_scan_plan(nq, n, k, sm_count, out.ctypes.data, m, C.byref(nc), C.byref(sm))
    return out, nc.value, sm.value


def scan_plan_pairs(nq: int, n: int, k: int, sm_count: int = 148):
    """The same for long rows (CTA pairs, 256-row tiles): (pieces[m,5], n_pairs, lists per query block)."""
    L = lib()
    nc, sm = C.c_int(0), C.c_int(0)
    m = L.nmslib_b200_scan_plan_pairs(nq, n, k, sm_count, None, 0, C.byref(nc), C.byref(sm))
    out = np.zeros((m, 5), np.int32)
    L.nmslib_b200_scan_plan_pairs(nq, n, k, sm_count, out.ctypes.data, m, C.byref(nc), C.byref(sm))
    return out, nc.value, sm.value


def set_option(name: str, value: int):
    """Process-wide variant selector (include/nmslib_b200.h: tc_pair, hnsw_team, force_exact, tc_split, u8_imma)."""
    _check(lib().nmslib_b200_set_option(name.encode(), int(value)))


def version() -> str:
    return lib().nmslib_b200_version().decode()
