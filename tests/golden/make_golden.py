"""Generate tests/golden/*.npz and *.hnsw from the UNMODIFIED reference.

Needs the reference compiled into oracle/_ref (a checkout of it at oracle/reference/, then
`make -C oracle ref`):

    python tests/golden/make_golden.py

Every fixture holds the inputs AND the reference's outputs, so a machine without the
reference can check both the oracle port and the CUDA path against
numbers produced by the reference itself.  Two routes are used on purpose:
  * "abi": the as-shipped C ABI of the reference (nmslib_index_create -> create_index on empty
    data -> add_data_point_batch -> initialize_pool -> knn_query_fill), i.e. exactly the call
    sequence lib.zig makes (SURVEY.md Appendix C);
  * "api": the public C++ API through oracle/ref_harness.cpp (needed for efSearch sweeps and
    SaveIndex, which the C ABI cannot do -- SURVEY.md 0.5).
"""
from __future__ import annotations

import ctypes as C
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
from oracle import oracle as O  # noqa: E402
from nmslib_zig_b200 import synth  # noqa: E402

OUT = Path(__file__).resolve().parent


# ---- the reference's C ABI, driven like lib.zig does --------------------------------------
class _Result(C.Structure):
    _fields_ = [("ids", C.POINTER(C.c_int32)), ("distances", C.POINTER(C.c_float)), ("size", C.c_size_t),
                ("capacity", C.c_size_t)]


_AF = C.CFUNCTYPE(C.c_void_p, C.c_size_t, C.c_void_p)
_FF = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p)


class _Alloc(C.Structure):
    _fields_ = [("alloc", _AF), ("free", _FF), ("ctx", C.c_void_p)]


_libc = C.CDLL(None)
_libc.malloc.restype = C.c_void_p
_libc.malloc.argtypes = [C.c_size_t]
_libc.free.argtypes = [C.c_void_p]
_ALLOC = _Alloc(_AF(lambda n, c: _libc.malloc(n)), _FF(lambda p, c: _libc.free(p)), None)


def ref_abi_knn(space, method, data, ids, queries, k, u8=False):
    L = C.CDLL(str(ROOT / "oracle" / "_ref" / "libnmslib_ref.so"))
    vp, sz = C.c_void_p, C.c_size_t
    L.nmslib_index_create.argtypes = [C.c_char_p, vp, C.c_char_p, C.c_int, C.c_int, C.POINTER(_Alloc), C.POINTER(vp)]
    L.nmslib_create_index.argtypes = [vp, vp, C.c_int]
    L.nmslib_add_data_point_batch.argtypes = [vp, vp, sz, sz, C.POINTER(C.c_int32), vp]
    L.nmslib_add_data_point_batch_uint8.argtypes = [vp, vp, sz, sz, C.POINTER(C.c_int32)]
    L.nmslib_initialize_pool.argtypes = [vp]
    L.nmslib_knn_query_fill.argtypes = [vp, vp, sz, sz, C.POINTER(_Result), sz]
    L.nmslib_index_destroy.argtypes = [vp]
    L.nmslib_init()
    h = vp()
    rc = L.nmslib_index_create(space.encode(), None, method.encode(), 2 if u8 else 0, 1 if u8 else 0,
                               C.byref(_ALLOC), C.byref(h))
    assert rc == 0, rc
    assert L.nmslib_create_index(h, None, 0) == 0  # lib.zig:629 -- on EMPTY data
    ids32 = np.ascontiguousarray(ids, np.int32)
    if u8:
        d = np.ascontiguousarray(data, np.uint8)
        assert L.nmslib_add_data_point_batch_uint8(h, d.ctypes.data, d.shape[0], d.shape[1],
                                                   ids32.ctypes.data_as(C.POINTER(C.c_int32))) == 0
        q = np.ascontiguousarray(queries, np.uint8)
    else:
        d = np.ascontiguousarray(data, np.float32)
        assert L.nmslib_add_data_point_batch(h, d.ctypes.data, d.shape[0], d.shape[1],
                                             ids32.ctypes.data_as(C.POINTER(C.c_int32)), None) == 0
        q = np.ascontiguousarray(queries, np.float32)
    L.nmslib_initialize_pool(h)  # lib.zig:802 / :892
    nq = q.shape[0]
    out_i = np.full((nq, k), -1, np.int32)
    out_d = np.full((nq, k), np.inf, np.float32)
    out_c = np.zeros(nq, np.int32)
    for i in range(nq):  # lib.zig:905-928
        r = _Result(out_i[i].ctypes.data_as(C.POINTER(C.c_int32)), out_d[i].ctypes.data_as(C.POINTER(C.c_float)), 0, k)
        rc = L.nmslib_knn_query_fill(h, q[i].ctypes.data, q.shape[1], k, C.byref(r), 0)
        assert rc == 0, rc
        out_c[i] = r.size
    L.nmslib_index_destroy(h)
    return out_i, out_d, out_c


def seq_case(name, space, data, queries, k, ids=None):
    n = data.shape[0]
    ids = np.arange(n, dtype=np.int32) if ids is None else np.asarray(ids, np.int32)
    u8 = space == "l2sqr_sift"
    # l2sqr is not a registered reference space (SURVEY 0.3): its golden distances come from the
    # reference's l2 path squared in float64 and rounded once; the ids are the l2 ids.
    ref_space = "l2" if space == "l2sqr" else space
    gi, gd, gc = ref_abi_knn(ref_space, "seq_search", data, ids, queries, k, u8=u8)
    ai, ad, ac = O.RefIndex(ref_space, "seq_search").add(data, ids).build("").knn(queries, k)
    # Both routes must agree.  Among exactly tied distances the reference orders by heap
    # address (knnqueue.h:73-74), which differs from run to run, so ids are compared only
    # where the distance is unique within the list.
    assert np.array_equal(gd, ad) and np.array_equal(gc, ac), name
    uniq = np.ones_like(gi, bool)
    uniq[:, 1:] &= gd[:, 1:] != gd[:, :-1]
    uniq[:, :-1] &= gd[:, :-1] != gd[:, 1:]
    uniq[:, -1] = False  # the k-th slot may hold any member of a tie group cut by k
    assert np.array_equal(gi[uniq], ai[uniq]), name
    np.savez_compressed(OUT / f"seq_{name}.npz", space=space, ref_space=ref_space, data=data, queries=queries,
                        ids=ids, k=k, ref_ids=gi, ref_dists=gd, ref_counts=gc)
    print(f"seq_{name}: n={n} dim={data.shape[1]} nq={queries.shape[0]} k={k}")


def hnsw_case(name, space, data, queries, k, params, efs, ids=None, keep_data=False, prefix="hnsw_"):
    n = data.shape[0]
    ids = np.arange(n, dtype=np.int32) if ids is None else np.asarray(ids, np.int32)
    r = O.RefIndex(space, "hnsw").add(data, ids).build(params)
    path = OUT / f"{prefix}{name}.hnsw"
    r.save(path)
    out = {"space": space, "queries": queries, "k": k, "efs": np.asarray(efs), "params": params}
    if keep_data:  # the regular (pointer-graph) index file carries no vectors (hnsw.cc:810-842)
        out["data"], out["ids"] = data, ids
    for ef in efs:
        r.set_query_params(f"efSearch={ef}")
        i, d, c = r.knn(queries, k)
        out[f"ids_ef{ef}"], out[f"dists_ef{ef}"], out[f"counts_ef{ef}"] = i, d, c
    # ground truth for recall: seq_search on the same data (SURVEY 8c)
    gi, gd, _ = O.RefIndex(space, "seq_search").add(data, ids).build("").knn(queries, k)
    out["exact_ids"], out["exact_dists"] = gi, gd
    np.savez_compressed(OUT / f"{prefix}{name}.npz", **out)
    print(f"{prefix}{name}: n={n} dim={data.shape[1]} file={path.stat().st_size} B")


def extra_spaces():
    """l1 / linf / angulardist over seq_search (SURVEY 8f N4); `make_golden.py extra` regenerates only these."""
    seq_case("l1_u128", "l1", synth.uniform(600, 128, 51) - 0.3, synth.uniform(16, 128, 52) - 0.3, 10)
    seq_case("l1_ragged19", "l1", synth.uniform(400, 19, 53), synth.uniform(12, 19, 54), 7, ids=np.arange(400) * 3 + 1)
    seq_case("linf_u64", "linf", synth.uniform(500, 64, 55) - 0.5, synth.uniform(16, 64, 56) - 0.5, 10)
    seq_case("angular_ragged37", "angulardist", synth.uniform(500, 37, 57) - 0.3, synth.uniform(16, 37, 58) - 0.3, 10)
    d = synth.uniform(200, 16, 59)
    d[50:60] = d[10:20]
    d[100] = 0.0
    q = np.concatenate([d[10:14], synth.uniform(4, 16, 60), np.zeros((1, 16), np.float32)])
    seq_case("angular_zero", "angulardist", d, q, 10)
    seq_case("l1_ties", "l1", d, q, 10)


def int_space_hnsw():
    """l2sqr_sift + hnsw: Hnsw<int> keeps the pointer graph and saves it with SaveRegularIndexBin (hnsw.cc:810-842); the
    searches are baseSearchAlgorithmV1Merge / Old (hnsw.cc:1076-1300).  `make_golden.py sift` regenerates only this."""
    hnsw_case("hnsw_sift", "l2sqr_sift", synth.sift_like_u8(3000, 47), synth.sift_like_u8(64, 48), 10,
              "M=8,efConstruction=100,indexThreadQty=1", [10, 50, 200, 1000], ids=np.arange(3000) * 2 + 5, keep_data=True,
              prefix="regular_")  # (not hnsw_*: the oracle's port of the search reads the optimized flat format only)


def main():
    assert O.ref_available(), "build oracle/_ref first: make -C oracle ref"
    if len(sys.argv) > 1 and sys.argv[1] == "extra":
        extra_spaces()
        return
    if len(sys.argv) > 1 and sys.argv[1] == "sift":
        int_space_hnsw()
        return
    int_space_hnsw()
    extra_spaces()
    rng = np.random.Generator(np.random.Philox(key=1234))

    # the reference's own pinned assertions (lib.zig:1292-1299): 3 unit vectors, ids 10/20/30
    seq_case("libzig_unit3", "l2", np.eye(4, dtype=np.float32)[:3], np.eye(4, dtype=np.float32)[:1], 2,
             ids=[10, 20, 30])
    # C1-shaped, reduced
    seq_case("l2_u128", "l2", synth.uniform(600, 128, 1), synth.uniform(24, 128, 2), 10)
    seq_case("l2sqr_sift128", "l2sqr", synth.sift_like_f32(700, 3), synth.sift_like_f32(16, 4), 10)
    seq_case("cos_ragged37", "cosinesimil", synth.uniform(500, 37, 11) - 0.3, synth.uniform(16, 37, 12) - 0.3, 10,
             ids=np.arange(500) * 7 + 3)
    seq_case("negdot_emb96", "negdotprod", synth.embedding_like(800, 96, 9), synth.embedding_like(12, 96, 10), 100)
    seq_case("sift_u8", "l2sqr_sift", synth.sift_like_u8(900, 7), synth.sift_like_u8(16, 8), 10)
    # exact ties (duplicated rows) and the cosine zero-norm branch
    d = synth.uniform(200, 16, 21)
    d[50:60] = d[10:20]
    d[100] = 0.0
    q = np.concatenate([d[10:14], synth.uniform(4, 16, 22), np.zeros((1, 16), np.float32)])
    seq_case("l2_ties", "l2", d, q, 10)
    seq_case("cos_zero", "cosinesimil", d, q, 10)
    du = synth.sift_like_u8(300, 23)
    du[100:120] = du[0:20]
    seq_case("sift_ties", "l2sqr_sift", du, du[:8], 12)
    # k > n
    seq_case("l2_k_gt_n", "l2", synth.uniform(7, 5, 31), synth.uniform(3, 5, 32), 10)

    # HNSW graphs built by the reference (M small so the files stay small)
    hnsw_case("l2_d32", "l2", synth.gist_like(2000, 32, 41, clusters=16), synth.gist_like(64, 32, 42, clusters=16), 10,
              "M=8,efConstruction=100,indexThreadQty=1", [10, 50, 200, 1000], ids=np.arange(2000) + 1000)
    hnsw_case("cos_d24", "cosinesimil", synth.gist_like(2000, 24, 43, clusters=16) - 0.2,
              synth.gist_like(64, 24, 44, clusters=16) - 0.2, 10, "M=8,efConstruction=100,indexThreadQty=1",
              [10, 50, 200])
    hnsw_case("negdot_d20", "negdotprod", synth.embedding_like(1500, 20, 45), synth.embedding_like(48, 20, 46), 10,
              "M=6,efConstruction=80,indexThreadQty=1", [20, 100])


if __name__ == "__main__":
    main()
