"""nmslib_b200_range_query_batch without a device: the symbol is exported and the whole batch is validated
before any work (the codes of nmslib_range_query_get_size / _fill), hnsw is refused like the single-query call."""
import ctypes as C

import numpy as np
import pytest

import nmslib_zig_b200 as nb
from nmslib_zig_b200 import index as nbi


def _index(method="seq_search", n=64, dim=8):
    idx = nb.Index("l2", None, method)
    idx.addDenseBatch(np.random.default_rng(0).random((n, dim), dtype=np.float32))
    return idx


def _call(idx, q, radii, results, nq=None, handle=True):
    L = nbi.lib()
    rp = radii.ctypes.data_as(C.POINTER(C.c_double)) if radii is not None else None
    return L.nmslib_b200_range_query_batch(idx.handle if handle else None, q.ctypes.data if q is not None else None,
                                           len(q) if nq is None else nq, 8, rp, results)


def _results(nq, cap=4):
    ids = np.zeros((nq, max(cap, 1)), np.int32)
    dists = np.zeros((nq, max(cap, 1)), np.float32)
    res = (nbi.Result * nq)()
    for i in range(nq):
        res[i] = nbi.Result(ids[i].ctypes.data_as(C.POINTER(C.c_int32)), dists[i].ctypes.data_as(C.POINTER(C.c_float)),
                            77, cap)
    return res, ids, dists


def test_symbol_is_exported():
    assert "nmslib_b200_range_query_batch" in nbi.EXT_SYMBOLS
    assert hasattr(nbi.lib(), "nmslib_b200_range_query_batch")
    assert [f for f, _ in nbi.Stats._fields_][-2:] == ["range_tc_queries", "range_fallback_queries"]


def test_invalid_arguments_are_rejected_before_any_work():
    idx = _index()
    q = np.zeros((3, 8), np.float32)
    radii = np.array([0.5, 1.0, 2.0])
    res, _, _ = _results(3)
    assert _call(idx, q, radii, res, handle=False) == 2
    assert _call(idx, None, radii, res, nq=3) == 2
    assert _call(idx, q, None, res) == 2
    assert _call(idx, q, radii, None) == 2
    assert _call(idx, q, radii, res, nq=0) == 2
    assert _call(idx, q, np.array([0.5, -1.0, 2.0]), res) == 2       # a negative radius anywhere
    res0, _, _ = _results(3)
    res0[2].capacity = 0
    assert _call(idx, q, radii, res0) == 2                            # a capacity of 0 anywhere
    resn, _, _ = _results(3)
    resn[1].ids = None
    assert _call(idx, q, radii, resn) == 2                            # a NULL result buffer anywhere
    idx.deinit()


def test_python_binding_validates_too():
    idx = _index()
    with pytest.raises(nb.NmslibError) as e:
        idx.rangeQueryBatch(np.zeros((2, 8), np.float32), [0.5, -0.5])
    assert e.value.code == 2
    with pytest.raises(nb.NmslibError) as e:
        idx.rangeQueryBatch(np.zeros((2, 8), np.float32), 0.5, capacity=0)
    assert e.value.code == 2
    r = idx.rangeQueryBatch(np.zeros((0, 8), np.float32), 0.5, capacity=7)
    assert r.ids.shape == (0, 0) and r.sizes.shape == (0,)
    idx.deinit()


def test_hnsw_is_space_incompatible():
    idx = _index("hnsw", n=200)
    idx.buildIndex(nb.Params({"M": 8, "efConstruction": 40, "b200_build": "host"}))
    with pytest.raises(nb.NmslibError) as e:
        idx.rangeQueryBatch(np.zeros((2, 8), np.float32), 0.5)
    assert e.value.code == 5
    idx.deinit()


def test_empty_sharded_index_answers_like_the_plain_index():
    """without a device an empty index fails the same way plain and under b200_devices (the check order of the
    single-query call: the device first, then the empty index)"""
    codes = []
    for params in (None, {"b200_devices": "0,0"}):
        idx = nb.Index("l2", None, "seq_search")
        idx.buildIndex(nb.Params(params) if params else None)
        try:
            idx.rangeQueryBatch(np.zeros((2, 8), np.float32), 0.5)
            codes.append(0)
        except nb.NmslibError as e:
            codes.append(e.code)
        idx.deinit()
    assert codes[0] == codes[1]
    if not nb.device_available():
        assert codes == [9, 9]
