"""CPU-side checks of the drop-in boundary: the shared library loads without a GPU, exports
every symbol include/nmslib_b200.h declares, and the non-compute entry points behave like the
reference shim (argument validation, error codes, ownership).  No kernel is launched here."""
import ctypes as C
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

import nmslib_zig_b200 as nb
from nmslib_zig_b200 import index as nbi

ROOT = Path(__file__).resolve().parents[1]


def _declared_symbols():
    text = (ROOT / "include" / "nmslib_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(nmslib_(?:b200_)?[a-z0-9_]+)\s*\(", text)))


def test_library_loads_and_exports_every_declared_symbol():
    L = nb.lib()
    declared = _declared_symbols()
    assert len([s for s in declared if not s.startswith("nmslib_b200_")]) == 37  # SURVEY 8b: 37 symbols
    out = subprocess.run(["nm", "-D", "--defined-only", str(nbi.LIB_PATH)], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (nmslib_[a-z0-9_]+)", out))
    missing = [s for s in declared if s not in exported]
    assert not missing, f"declared but not exported: {missing}"
    assert sorted(nbi.ABI_SYMBOLS + nbi.EXT_SYMBOLS) == declared
    for s in declared:
        getattr(L, s)


def test_reference_header_symbols_are_all_present():
    """The 37 names the reference exports (SURVEY 8b list, probed with nm -D on the reference)."""
    ref = ("nmslib_init nmslib_index_create nmslib_index_destroy nmslib_create_index nmslib_reset_index "
           "nmslib_create_params nmslib_add_param nmslib_free_params nmslib_get_space_type nmslib_get_method "
           "nmslib_free_string nmslib_get_last_error_detail nmslib_add_data_point nmslib_add_data_point_batch "
           "nmslib_add_data_point_batch_uint8 nmslib_add_data_point_batch_string nmslib_add_data_point_batch_pointers "
           "nmslib_knn_query_get_size nmslib_knn_query_fill nmslib_knn_query_batch nmslib_range_query_get_size "
           "nmslib_range_query_fill nmslib_get_distance nmslib_get_data_point_size nmslib_get_data_point_fill "
           "nmslib_get_data_point_string nmslib_borrow_data_dense nmslib_borrow_data_sparse nmslib_save_index "
           "nmslib_load_index nmslib_set_query_time_params nmslib_set_thread_pool_size nmslib_get_thread_pool_size "
           "nmslib_data_qty nmslib_index_memory_usage nmslib_initialize_pool nmslib_free_result").split()
    assert len(ref) == 37
    assert sorted(ref) == sorted(nbi.ABI_SYMBOLS)


def test_struct_layouts_match_the_abi():
    assert C.sizeof(nbi.Result) == 32 and nbi.Result.size.offset == 16 and nbi.Result.capacity.offset == 24
    assert C.sizeof(nbi.Allocator) == 24
    assert C.sizeof(nbi.ErrorDetail) == 32


def test_version_string_names_the_arch():
    assert "sm_100a" in nb.version()


def test_dense_workflow_metadata_like_lib_zig_test(tmp_path):
    """lib.zig:1273-1313 minus the query (no GPU here): counts, names, getDistance, getDataPoint,
    save -> reset -> load."""
    before = nb.live_allocations()
    idx = nb.Index.init("l2", nb.Params({"dim": 4}), "seq_search", "DenseVector", "Float")
    data = np.eye(4, dtype=np.float32)[:3]
    idx.addDenseBatch(data, [10, 20, 30])
    idx.buildIndex(None, False)
    assert idx.dataQty() == 3
    assert idx.getSpaceType() == "l2" and idx.getMethod() == "seq_search"
    assert abs(idx.getDistance(0, 1) - np.sqrt(2.0)) < 1e-6       # lib.zig:1419-1424
    assert np.array_equal(idx.getDataPoint(0), data[0])
    assert np.array_equal(idx.borrowDataDense(1), data[1])
    assert idx.memoryUsage() == 3 * (16 + 16) + 3 * 4 * 4            # nmslib_c.cpp:1546-1565
    idx.save(str(tmp_path / "test_index"), True)
    idx.reset()
    assert idx.dataQty() == 0
    loaded = nb.Index.load(str(tmp_path / "test_index"), "DenseVector", "Float", True)
    assert loaded.dataQty() == 3
    assert np.array_equal(loaded.getDataPoint(0), data[0])
    loaded.deinit()
    idx.deinit()
    assert nb.live_allocations() == before, "allocator callbacks leaked (std.testing.allocator would fail)"


def test_error_codes_match_the_reference_conventions():
    with pytest.raises(nb.NmslibError) as e:
        nb.Index("l2sqr_sift", None, "seq_search", "DenseVector", "Float")   # space / data type mismatch
    assert e.value.name == "SpaceIncompatible"
    with pytest.raises(nb.NmslibError) as e:
        nb.Index("jaccard_sparse", None, "hnsw", "SparseVector", "Float")    # stays on the reference CPU code
    assert e.value.name == "SpaceIncompatible"
    idx = nb.Index("cosine", None, "hnsw")                                    # lib.zig:530-533 alias
    assert idx.getSpaceType() == "cosinesimil"
    with pytest.raises(nb.NmslibError) as e:
        idx.buildIndex(nb.Params({"bogus": 1}))                               # CheckUnused -> error 8
    assert e.value.name == "IndexBuildFailed"
    idx.buildIndex(nb.Params({"M": 16, "efConstruction": 200}))
    with pytest.raises(nb.NmslibError) as e:
        idx.setQueryTimeParams(nb.Params({"ef": 10, "efSearch": 20}))         # hnsw.cc:478-480
    assert e.value.name == "InvalidArgument"
    idx.setQueryTimeParams(nb.Params({"efSearch": 50, "algoType": "v1merge"}))
    with pytest.raises(nb.NmslibError) as e:
        idx.rangeQuery(np.zeros(4, np.float32), 1.0)                          # lib.zig:1452-1456 accepts this
    assert e.value.name == "SpaceIncompatible"
    with pytest.raises(nb.NmslibError) as e:
        idx.addDenseBatch(np.zeros((2, 4), np.float32))
        idx.addDenseBatch(np.zeros((2, 5), np.float32))                       # dimension fixed by the first row
    assert e.value.name == "InvalidArgument"
    idx.deinit()
    other = nb.Index("l2", None, "vptree")
    with pytest.raises(nb.NmslibError) as e:
        other.buildIndex()
    assert e.value.name == "IndexBuildFailed"
    other.deinit()


def test_raw_abi_argument_validation():
    L = nb.lib()
    n = C.c_size_t()
    q = np.zeros(4, np.float32)
    assert L.nmslib_knn_query_get_size(None, q.ctypes.data, 4, 10, C.byref(n), 0) == 2
    idx = nb.Index("l2", None, "seq_search")
    assert L.nmslib_knn_query_get_size(idx.handle, q.ctypes.data, 4, 0, C.byref(n), 0) == 2   # k == 0
    assert L.nmslib_knn_query_get_size(idx.handle, q.ctypes.data, 4, 7, C.byref(n), 0) == 0 and n.value == 7
    ids = np.zeros(3, np.int32)
    d = np.zeros(3, np.float32)
    res = nbi.Result(ids.ctypes.data_as(C.POINTER(C.c_int32)), d.ctypes.data_as(C.POINTER(C.c_float)), 0, 3)
    assert L.nmslib_knn_query_fill(idx.handle, q.ctypes.data, 4, 3, C.byref(res), 0) == 8      # not built
    assert L.nmslib_knn_query_fill(idx.handle, q.ctypes.data, 4, 0, C.byref(res), 0) == 2      # k == 0 (Q8)
    assert L.nmslib_set_thread_pool_size(idx.handle, 0) == 2
    assert L.nmslib_set_thread_pool_size(idx.handle, 8) == 0 and L.nmslib_get_thread_pool_size(idx.handle) == 8
    assert L.nmslib_data_qty(None) == 0
    idx.deinit()


def test_uint8_ingest_requires_128_dims():
    idx = nb.Index("l2sqr_sift", None, "seq_search", "DenseUInt8Vector", "Int")
    with pytest.raises(nb.NmslibError):
        idx.addUInt8Batch(np.zeros((2, 64), np.uint8))                        # space_l2sqr_sift.cc:137
    idx.addUInt8Batch(np.full((2, 128), 3, np.uint8))
    idx.buildIndex()
    assert idx.getDistance(0, 1) == 0.0
    assert idx.getDataPoint(1).dtype == np.uint8
    idx.deinit()


def test_hnsw_file_import_and_rewrite_is_byte_identical(golden_dir, tmp_path):
    """The optimized-index reader/writer round-trips a file written by the reference
    (hnsw.cc:774-806) byte for byte."""
    src = golden_dir / "hnsw_l2_d32.hnsw"
    idx = nb.Index.load(str(src))
    assert idx.getMethod() == "hnsw" and idx.getSpaceType() == "l2" and idx.dataQty() == 2000
    out = tmp_path / "rewritten.hnsw"
    idx.save(str(out), False)
    assert out.read_bytes() == src.read_bytes()
    idx.deinit()
    cos = nb.Index.load(str(golden_dir / "hnsw_cos_d24.hnsw"))
    assert cos.getSpaceType() == "cosinesimil"      # SURVEY Q11: read dist_func_type_ from the header
    v = cos.getDataPoint(5)
    assert abs(float(np.dot(v, v)) - 1.0) < 1e-5     # cosine rows are stored normalised (hnsw.cc:441-446)
    cos.deinit()


def test_sharding_entry_points_validate_without_a_device():
    """include/nmslib_b200.h section "row-sharded multi-GPU search": argument validation and the b200_devices parser
    need no GPU; anything that would touch a device fails loudly (there is no CPU fallback)."""
    text = (ROOT / "include" / "nmslib_b200.h").read_text()
    assert "#define NMSLIB_B200_SHARD_BLOB_BYTES 256" in text
    idx = nb.Index("l2", None, "seq_search")
    idx.addDenseBatch(np.eye(4, dtype=np.float32))
    for bad in ("0,,1", "x", "3-1", "-1"):
        with pytest.raises(nb.NmslibError) as e:
            idx.buildIndex(nb.Params({"b200_devices": bad}))
        assert e.value.name == "IndexBuildFailed"
    idx.buildIndex(nb.Params({"b200_devices": "0"}))          # one device: an ordinary index
    with pytest.raises(nb.NmslibError):
        idx.shardConnect(0, 2, b"\0" * 512)                    # no exported window
    if not nb.device_available():
        with pytest.raises(nb.NmslibError):
            idx.shardExport(16, 4)
    idx.deinit()
    hn = nb.Index("l2", None, "hnsw")
    hn.addDenseBatch(np.eye(4, dtype=np.float32))
    # hnsw: replicas of the graph, queries split (SURVEY 8e); where devices are visible the list must name existing ones
    hn.buildIndex(nb.Params({"b200_devices": "0,0" if nb.device_available() else "0,1"}))
    with pytest.raises(nb.NmslibError):
        hn.buildIndex(nb.Params({"b200_devices": "0,,1"}))
    if not nb.device_available():
        with pytest.raises(nb.NmslibError):                    # no device: the query fails, nothing falls back to the host
            hn.knnQueryBatch(np.eye(4, dtype=np.float32), 2)
    hn.deinit()
    with pytest.raises(nb.NmslibError):
        nb.set_option("no_such_option", 1)
    nb.set_option("tc_pair", 1)
