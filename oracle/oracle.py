"""oracle/oracle.py -- TEST INFRASTRUCTURE ONLY.

ctypes loaders for (a) liboracle_knn.so, the plain-C restatement of the reference's
query path (knn_oracle.c), and (b) oracle/_ref/*.so, the UNMODIFIED reference compiled
by oracle/Makefile from a checkout of it at oracle/reference/.  Imported only by tests/, by
__graft_entry__.smoke() and by bench.py's cpu_baseline / --impl reference legs; the
product package never imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
SPACE_CODES = {"l2": 0, "l2sqr": 1, "cosinesimil": 2, "cosine": 2, "negdotprod": 3, "l2sqr_sift": 4, "l1": 5, "linf": 6,
               "angulardist": 7}

_i32p = C.POINTER(C.c_int32)
_f32p = C.POINTER(C.c_float)
_i64p = C.POINTER(C.c_int64)


def _ptr(a, typ):
    return a.ctypes.data_as(typ) if a is not None else None


def build() -> None:
    """Compile the C restatement and, where a checkout of the reference sits at oracle/reference/, oracle/_ref."""
    subprocess.run(["make", "-s", "-C", str(HERE), f"-j{os.cpu_count() or 4}", "oracle", "ref"], check=True)


# --------------------------------------------------------------------------- C restatement
_port = None


def port():
    global _port
    if _port is None:
        so = HERE / "liboracle_knn.so"
        if not so.exists():
            build()
        L = C.CDLL(str(so))
        for name in ("orc_l2sqr", "orc_l2", "orc_norm_scalar_product", "orc_cosine", "orc_negdot",
                     "orc_hnsw_l2sqr", "orc_hnsw_dot", "orc_l1", "orc_linf", "orc_angular"):
            f = getattr(L, name)
            f.restype = C.c_float
            f.argtypes = [_f32p, _f32p, C.c_size_t]
        L.orc_l2sqr_sift.restype = C.c_int32
        L.orc_l2sqr_sift.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_seq_knn.restype = C.c_int
        L.orc_seq_knn.argtypes = [C.c_int, C.c_void_p, C.c_size_t, C.c_size_t, _i32p, C.c_void_p,
                                  C.c_size_t, C.c_size_t, _i32p, _f32p, _i32p, C.c_int]
        L.orc_hnsw_load.restype = C.c_void_p
        L.orc_hnsw_load.argtypes = [C.c_char_p]
        L.orc_hnsw_free.argtypes = [C.c_void_p]
        L.orc_hnsw_info.argtypes = [C.c_void_p] + [C.POINTER(C.c_uint64)] * 4 + [
            _i32p, C.POINTER(C.c_uint32), _i32p]
        L.orc_hnsw_knn.restype = C.c_int
        L.orc_hnsw_knn.argtypes = [C.c_void_p, _f32p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t,
                                   C.c_int, _i32p, _f32p, _i32p, _i64p, C.c_int]
        L.orc_max_threads.restype = C.c_int
        _port = L
    return _port


def pair_distance(space: str, a: np.ndarray, b: np.ndarray):
    """distance(data point a, query b) exactly as the seq_search path computes it."""
    L = port()
    if space == "l2sqr_sift":
        a = np.ascontiguousarray(a, np.uint8)
        b = np.ascontiguousarray(b, np.uint8)
        return int(L.orc_l2sqr_sift(a.ctypes.data, b.ctypes.data))
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    fn = {"l2": L.orc_l2, "l2sqr": L.orc_l2sqr, "cosinesimil": L.orc_cosine, "cosine": L.orc_cosine,
          "negdotprod": L.orc_negdot, "hnsw_l2sqr": L.orc_hnsw_l2sqr, "hnsw_dot": L.orc_hnsw_dot,
          "l1": L.orc_l1, "linf": L.orc_linf, "angulardist": L.orc_angular}[space]
    return float(fn(_ptr(a, _f32p), _ptr(b, _f32p), a.size))


def seq_knn(space: str, data: np.ndarray, queries: np.ndarray, k: int, ids=None, threads: int = 0):
    """Sequential-search kNN (seqsearch.cc:144-150).  Returns (ids[nq,k], dists[nq,k], counts[nq])."""
    L = port()
    dt = np.uint8 if space == "l2sqr_sift" else np.float32
    data = np.ascontiguousarray(data, dt)
    queries = np.ascontiguousarray(queries, dt)
    n, dim = data.shape if data.ndim == 2 else (0, queries.shape[1])
    nq = queries.shape[0]
    out_i = np.full((nq, k), -1, np.int32)
    out_d = np.full((nq, k), np.inf, np.float32)
    out_c = np.zeros(nq, np.int32)
    ids_a = None if ids is None else np.ascontiguousarray(ids, np.int32)
    rc = L.orc_seq_knn(SPACE_CODES[space], data.ctypes.data, n, dim, _ptr(ids_a, _i32p),
                       queries.ctypes.data, nq, k, _ptr(out_i, _i32p), _ptr(out_d, _f32p),
                       _ptr(out_c, _i32p), threads or L.orc_max_threads())
    if rc != 0:
        raise RuntimeError(f"orc_seq_knn failed rc={rc}")
    return out_i, out_d, out_c


class PortHnsw:
    """The C restatement of Hnsw::Search over a file written by Hnsw::SaveIndex."""

    def __init__(self, path: str):
        self.L = port()
        self.h = self.L.orc_hnsw_load(str(path).encode())
        if not self.h:
            raise RuntimeError(f"cannot parse optimized HNSW index {path}")
        t, d, m, m0 = (C.c_uint64() for _ in range(4))
        ml, df = C.c_int32(), C.c_int32()
        ep = C.c_uint32()
        self.L.orc_hnsw_info(self.h, t, d, m, m0, ml, ep, df)
        self.total, self.dim, self.maxM, self.maxM0 = t.value, d.value, m.value, m0.value
        self.maxlevel, self.enterpoint, self.dist_func = ml.value, ep.value, df.value

    def knn(self, queries, k, ef, algo="hybrid", threads=0):
        q = np.ascontiguousarray(queries, np.float32)
        nq = q.shape[0]
        out_i = np.full((nq, k), -1, np.int32)
        out_d = np.full((nq, k), np.inf, np.float32)
        out_c = np.zeros(nq, np.int32)
        ev = np.zeros(nq, np.int64)
        rc = self.L.orc_hnsw_knn(self.h, _ptr(q, _f32p), nq, q.shape[1], k, ef,
                                 {"hybrid": 0, "v1merge": 1, "old": 2}[algo], _ptr(out_i, _i32p),
                                 _ptr(out_d, _f32p), _ptr(out_c, _i32p), _ptr(ev, _i64p),
                                 threads or self.L.orc_max_threads())
        if rc != 0:
            raise RuntimeError(f"orc_hnsw_knn rc={rc}")
        return out_i, out_d, out_c, ev

    def close(self):
        if self.h:
            self.L.orc_hnsw_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# --------------------------------------------------------------------------- the real reference
def ref_available() -> bool:
    return (HERE / "_ref" / "libref_harness.so").exists() and (HERE / "_ref" / "libnmslib_ref.so").exists()


_harness = None


def harness():
    global _harness
    if _harness is None:
        C.CDLL(str(HERE / "_ref" / "libnmslib_ref.so"), mode=C.RTLD_GLOBAL)
        L = C.CDLL(str(HERE / "_ref" / "libref_harness.so"))
        L.refh_open.restype = C.c_void_p
        L.refh_open.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
        L.refh_close.argtypes = [C.c_void_p]
        L.refh_add_f32.argtypes = [C.c_void_p, _f32p, C.c_size_t, C.c_size_t, _i32p]
        L.refh_add_u8.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, _i32p]
        L.refh_build.argtypes = [C.c_void_p, C.c_char_p]
        L.refh_set_query_params.argtypes = [C.c_void_p, C.c_char_p]
        L.refh_knn_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t,
                                     _i32p, _f32p, _i32p, C.c_int]
        L.refh_save.argtypes = [C.c_void_p, C.c_char_p]
        if hasattr(L, "refh_load"):
            L.refh_load.argtypes = [C.c_void_p, C.c_char_p]
        L.refh_size.restype = C.c_size_t
        L.refh_size.argtypes = [C.c_void_p]
        L.refh_last_error.restype = C.c_char_p
        L.refh_last_error.argtypes = [C.c_void_p]
        L.refh_max_threads.restype = C.c_int
        _harness = L
    return _harness


class RefIndex:
    """The unmodified reference driven through its public C++ API (ref_harness.cpp)."""

    def __init__(self, space: str, method: str):
        self.L = harness()
        self.space, self.method = space, method
        self.u8 = space == "l2sqr_sift"
        self.h = self.L.refh_open(space.encode(), method.encode(), int(self.u8))
        if not self.h:
            raise RuntimeError(f"reference cannot create space {space}")

    def _chk(self, rc, what):
        if rc != 0:
            raise RuntimeError(f"reference {what} failed rc={rc}: {self.L.refh_last_error(self.h).decode()}")

    def add(self, data, ids=None):
        ids_a = None if ids is None else np.ascontiguousarray(ids, np.int32)
        if self.u8:
            d = np.ascontiguousarray(data, np.uint8)
            self._chk(self.L.refh_add_u8(self.h, d.ctypes.data, d.shape[0], _ptr(ids_a, _i32p)), "add")
        else:
            d = np.ascontiguousarray(data, np.float32)
            self._chk(self.L.refh_add_f32(self.h, _ptr(d, _f32p), d.shape[0], d.shape[1],
                                          _ptr(ids_a, _i32p)), "add")
        return self

    def build(self, params: str = ""):
        self._chk(self.L.refh_build(self.h, params.encode()), "build")
        return self

    def set_query_params(self, params: str):
        self._chk(self.L.refh_set_query_params(self.h, params.encode()), "set_query_params")
        return self

    def knn(self, queries, k, threads=1):
        q = np.ascontiguousarray(queries, np.uint8 if self.u8 else np.float32)
        nq, dim = q.shape
        out_i = np.full((nq, k), -1, np.int32)
        out_d = np.full((nq, k), np.inf, np.float32)
        out_c = np.zeros(nq, np.int32)
        self._chk(self.L.refh_knn_batch(self.h, q.ctypes.data, nq, dim, k, _ptr(out_i, _i32p),
                                        _ptr(out_d, _f32p), _ptr(out_c, _i32p), threads), "knn")
        return out_i, out_d, out_c

    def save(self, path):
        self._chk(self.L.refh_save(self.h, str(path).encode()), "save")

    def load(self, path):
        """Index::LoadIndex of an optimized HNSW file (e.g. one written by nmslib_b200's nmslib_save_index)."""
        self._chk(self.L.refh_load(self.h, str(path).encode()), "load")
        return self

    def max_threads(self):
        return int(self.L.refh_max_threads())

    def close(self):
        if self.h:
            self.L.refh_close(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def regular_to_flat_hnsw(regular_path, data: np.ndarray, ids, out_path):
    """TEST INFRASTRUCTURE.  Rewrite the reference's REGULAR index file (Hnsw::SaveRegularIndexBin, hnsw.cc:810-842:
    links of the pointer graph, what Hnsw<int> = l2sqr_sift + hnsw saves) plus its uint8 data set as an optimized flat
    file (hnsw.cc:774-806) with the rows widened to float: the C port of the flat search then walks the same graph
    with distances that are exact integers in fp32 -- the claim the device path makes for SURVEY row a18
    (baseSearchAlgorithmV1Merge / Old, hnsw.cc:1076-1300, use the same beam rule as the flat searches)."""
    import struct
    raw = Path(regular_path).read_bytes()
    flag, total, maxlevel, enter = struct.unpack_from("<IIiI", raw, 0)
    M, maxM, maxM0 = struct.unpack_from("<QQQ", raw, 16)
    assert flag == 0 and total == data.shape[0]
    pos = 40
    dim = data.shape[1]
    vec = np.ascontiguousarray(data, np.float32)
    ids = np.ascontiguousarray(ids, np.int32)
    off0 = 16 + 4 * dim
    mem = off0 + 4 * (maxM0 + 1)
    recs = bytearray(b"\x01" * (mem * total))
    uppers = []
    levels = []
    for i in range(total):
        level, = struct.unpack_from("<I", raw, pos)
        pos += 4
        levels.append(level)
        up = bytearray()
        for l in range(level + 1):
            cnt, = struct.unpack_from("<I", raw, pos)
            pos += 4
            fr = raw[pos:pos + 4 * cnt]
            pos += 4 * cnt
            if l == 0:
                struct.pack_into("<i", recs, i * mem + off0, cnt)
                recs[i * mem + off0 + 4:i * mem + off0 + 4 + 4 * cnt] = fr
            else:
                blk = bytearray(4 * (maxM + 1))
                struct.pack_into("<i", blk, 0, cnt)
                blk[4:4 + 4 * cnt] = fr
                up += blk
        struct.pack_into("<iiQ", recs, i * mem, int(ids[i]), -1, 4 * dim)
        recs[i * mem + 16:i * mem + 16 + 4 * dim] = vec[i].tobytes()
        uppers.append(bytes(up))
    maxlevel = min(maxlevel, levels[enter]) if total else maxlevel   # the pointer search starts at enterpoint_->level
    with open(out_path, "wb") as f:
        f.write(struct.pack("<IIQQQiIQQiQ", 1, total, mem, off0, 0, maxlevel, enter, maxM, maxM0, 1 if dim % 16 == 0 else 2, 3))
        f.write(recs)
        for up in uppers:
            f.write(struct.pack("<I", len(up)))
            f.write(up)
    return out_path
