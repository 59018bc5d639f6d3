"""uint8 (l2sqr_sift) HNSW on byte rows: the beam search reads 128-byte rows and computes every distance as an exact
integer, so the answers equal those of widened fp32 rows and of the C port bit for bit (ids and distance bits)."""
from __future__ import annotations

import os
import struct
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np
import pytest

import nmslib_zig_b200 as nb
from nmslib_zig_b200 import synth
from oracle import oracle as O
from helpers import assert_knn_matches, count_mismatches

pytestmark = pytest.mark.gpu

GOLDEN = Path(__file__).resolve().parent / "golden"
ROOT = Path(__file__).resolve().parents[1]


def bits(a):
    return np.asarray(a, np.float32).view(np.int32)


def assert_same(a_ids, a_d, b_ids, b_d, what):
    assert np.array_equal(a_ids, b_ids), f"{what}: ids differ"
    assert np.array_equal(bits(a_d), bits(b_d)), f"{what}: distance bits differ"


def device_knn(idx, q, k):
    import torch
    d_q = torch.from_numpy(np.ascontiguousarray(q, np.uint8)).cuda()
    ids = torch.empty((len(q), k), dtype=torch.int32, device="cuda")
    dd = torch.empty((len(q), k), dtype=torch.float32, device="cuda")
    idx.knnDevice(d_q.data_ptr(), len(q), q.shape[1], k, ids.data_ptr(), dd.data_ptr())
    torch.cuda.synchronize()
    return ids.cpu().numpy(), dd.cpu().numpy()


def write_dat(path, data, ids):
    with open(str(path) + ".dat", "wb") as f:
        f.write(struct.pack("<Q", len(data)))
        for row, i in zip(np.asarray(data, np.uint8), np.asarray(ids, np.int32)):
            f.write(struct.pack("<QiiQ", 148, int(i), -1, 132))
            f.write(row.tobytes())
            f.write(struct.pack("<i", int(np.sum(row.astype(np.int64) ** 2))))


def set_ef(idx, ef):
    idx.setQueryTimeParams(nb.Params({"efSearch": int(ef)}))


def port_answers(regular_path, data, ids, q, k, ef, tmp):
    port = O.PortHnsw(O.regular_to_flat_hnsw(regular_path, data, ids, Path(tmp) / "flat.hnsw"))
    out = port.knn(np.asarray(q, np.float32), k, ef)[:3]
    port.close()
    return out


def test_golden_graph_device_entry_and_loaded_index_equal_the_host_entry(tmp_path):
    g = np.load(GOLDEN / "regular_hnsw_sift.npz")
    data, ids, q = g["data"], g["ids"], g["queries"]
    imp = nb.Index("l2sqr_sift", None, "hnsw", "DenseUInt8Vector", "Int")
    imp.addUInt8Batch(data, ids)
    imp.importHnsw(GOLDEN / "regular_hnsw_sift.hnsw")
    src = tmp_path / "golden.hnsw"
    src.write_bytes((GOLDEN / "regular_hnsw_sift.hnsw").read_bytes())
    write_dat(src, data, ids)
    loaded = nb.Index.load(str(src), "DenseUInt8Vector", "Int")
    for ef in g["efs"]:
        set_ef(imp, ef)
        set_ef(loaded, ef)
        h = imp.knnQueryBatch(q, 10)
        di, dd = device_knn(imp, q, 10)
        assert_same(di, dd, h.ids, h.distances, f"device entry ef={ef}")
        l = loaded.knnQueryBatch(q, 10)
        assert_same(l.ids, l.distances, h.ids, h.distances, f"loaded index ef={ef}")
        li, ld = device_knn(loaded, q, 10)
        assert_same(li, ld, h.ids, h.distances, f"loaded index, device entry ef={ef}")
        same = h.ids == g[f"ids_ef{ef}"]                     # the reference's distances where the ids agree
        assert np.array_equal(bits(h.distances[same]), bits(g[f"dists_ef{ef}"][same]))
    imp.deinit()
    loaded.deinit()


def device_built_case():
    n = 40_000
    data = synth.sift_like_u8(n, 21)
    data[1000:1100] = data[0:100]                            # duplicated rows
    data[20_000] = data[5]
    data[777] = 0                                            # one all-zero row
    ids = np.arange(n, dtype=np.int32) * 7 + 3
    q = synth.sift_like_u8(257, 22)
    q[0] = data[5]
    q[1] = 0
    q[2] = data[1050]
    return data, ids, q


def test_device_built_graph_equals_widened_rows_bit_for_bit(tmp_path):
    """A graph built on the device (auto from 16 384 rows), saved as a regular file: the byte rows answer exactly like an
    l2 index holding the same values as floats over the same graph (the fp32 kernel), and like the C port up to the
    order of equal distances inside the beam."""
    data, ids, q = device_built_case()
    idx = nb.Index("l2sqr_sift", None, "hnsw", "DenseUInt8Vector", "Int")
    idx.addUInt8Batch(data, ids)
    idx.buildIndex(nb.Params({"M": 16, "efConstruction": 100}))
    path = tmp_path / "dev.hnsw"
    idx.save(str(path))
    wide = nb.Index("l2", None, "hnsw")
    wide.addDenseBatch(data.astype(np.float32), ids)
    wide.importHnsw(path)
    port = O.PortHnsw(O.regular_to_flat_hnsw(path, data, ids, tmp_path / "flat.hnsw"))
    qf = q.astype(np.float32)
    for ef in (10, 50, 200, 1000):
        set_ef(idx, ef)
        set_ef(wide, ef)
        for k in (1, 10, 100):
            h = idx.knnQueryBatch(q, k)
            w = wide.knnQueryBatch(qf, k)
            assert_same(h.ids, h.distances, w.ids, w.distances, f"byte vs fp32 rows ef={ef} k={k}")
            di, dd = device_knn(idx, q, k)
            assert_same(di, dd, h.ids, h.distances, f"device ef={ef} k={k}")
            # Integer distances tie often.  The port's SortArrBI insertion places a new item before equal keys where
            # the kernel places it after, so a query whose beam meets such a tie may expand another node: a few
            # queries differ, every other one matches exactly.
            pi, pd, pc, _ = port.knn(qf, k, ef)
            bad = count_mismatches(h.ids, h.distances, h.sizes, pi, pd, pc, exact=True)
            assert bad <= len(q) // 20, f"ef={ef} k={k}: {bad} of {len(q)} queries differ from the C port"
    for i in range(0, len(q), 16):                           # reported distances are the exact integer distances
        pos = (h.ids[i] - 3) // 7
        want = np.sum((data[pos].astype(np.int64) - q[i].astype(np.int64)) ** 2, axis=1)
        assert np.array_equal(h.distances[i].astype(np.int64), want)
    port.close()
    wide.deinit()
    idx.deinit()


def test_team_kernels_are_bit_identical_to_the_one_warp_kernel(tmp_path):
    script = (
        "import sys, numpy as np\n"
        f"sys.path.insert(0, {str(ROOT)!r})\n"
        "import nmslib_zig_b200 as nb\n"
        "from nmslib_zig_b200 import synth\n"
        "nb.set_option('hnsw_team', int(sys.argv[2]))\n"
        "data, q = synth.sift_like_u8(20000, 31), synth.sift_like_u8(700, 32)\n"
        "idx = nb.Index('l2sqr_sift', None, 'hnsw', 'DenseUInt8Vector', 'Int'); idx.addUInt8Batch(data)\n"
        "idx.buildIndex(nb.Params({'M': 16, 'efConstruction': 100, 'b200_build': 'host', 'indexThreadQty': 1}))\n"
        "idx.save(sys.argv[1] + '.hnsw')\n"
        "out = []\n"
        "for ef in (10, 64, 300, 1000):\n"
        "    idx.setQueryTimeParams(nb.Params({'efSearch': ef}))\n"
        "    r = idx.knnQueryBatch(q, 10); out += [r.ids, r.distances.view(np.int32)]\n"
        "np.save(sys.argv[1], np.stack(out))\n")
    outs, graphs = [], []
    for mode in ("0", "2", "4"):
        path = tmp_path / f"team{mode}.npy"
        subprocess.run([sys.executable, "-c", script, str(path), mode], check=True, timeout=900)
        outs.append(np.load(path))
        graphs.append((tmp_path / f"team{mode}.npy.hnsw").read_bytes())
    assert graphs[0] == graphs[1] == graphs[2]                # (the same graph in each process)
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])


def _replicas_match_plain_index(devices):
    n, nq, k = 6000, 301, 10
    data, q = synth.sift_like_u8(n, 41), synth.sift_like_u8(nq, 42)
    ext = np.arange(n, dtype=np.int32) * 2 + 11
    grp = nb.Index("l2sqr_sift", None, "hnsw", "DenseUInt8Vector", "Int")
    grp.addUInt8Batch(data, ext)
    grp.buildIndex(nb.Params({"M": 12, "efConstruction": 80, "b200_build": "host", "b200_devices": devices}))
    set_ef(grp, 64)
    b = grp.knnQueryBatch(q, k)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "g.hnsw")
        grp.save(path)                                       # the graph the replicas search
        one = nb.Index.load(path, "DenseUInt8Vector", "Int")
    set_ef(one, 64)
    a = one.knnQueryBatch(q, k)
    assert_same(a.ids, a.distances, b.ids, b.distances, f"replicas {devices}")
    assert np.array_equal(a.sizes, b.sizes)
    set_ef(grp, 200)
    set_ef(one, 200)
    a, b = one.knnQueryBatch(q[:50], k), grp.knnQueryBatch(q[:50], k)
    assert_same(a.ids, a.distances, b.ids, b.distances, f"replicas {devices} ef=200")
    one.deinit()
    grp.deinit()


def test_replicas_on_one_device_match_plain_index():
    _replicas_match_plain_index("0,0")


def test_replicas_on_two_devices_match_plain_index():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _replicas_match_plain_index("0,1")


def test_byte_rows_take_a_quarter_of_the_device_bytes():
    g = np.load(GOLDEN / "regular_hnsw_sift.npz")
    data, ids = g["data"], g["ids"]
    u8 = nb.Index("l2sqr_sift", None, "hnsw", "DenseUInt8Vector", "Int")
    u8.addUInt8Batch(data, ids)
    u8.importHnsw(GOLDEN / "regular_hnsw_sift.hnsw")
    f32 = nb.Index("l2", None, "hnsw")
    f32.addDenseBatch(data.astype(np.float32), ids)
    f32.importHnsw(GOLDEN / "regular_hnsw_sift.hnsw")
    q = g["queries"]
    a, b = u8.knnQueryBatch(q, 10), f32.knnQueryBatch(q.astype(np.float32), 10)
    assert_same(a.ids, a.distances, b.ids, b.distances, "uint8 vs float rows")
    saved = f32.stats()["device_bytes"] - u8.stats()["device_bytes"]
    assert saved >= len(data) * 384, saved
    u8.deinit()
    f32.deinit()


def test_appended_rows_small_indexes_wide_beams_and_bad_queries(tmp_path):
    data = synth.sift_like_u8(3000, 51)
    more = synth.sift_like_u8(500, 52)
    q = synth.sift_like_u8(64, 53)
    idx = nb.Index("l2sqr_sift", None, "hnsw", "DenseUInt8Vector", "Int")
    idx.addUInt8Batch(data)
    idx.buildIndex(nb.Params({"M": 10, "efConstruction": 60, "b200_build": "host", "indexThreadQty": 1}))
    idx.knnQueryBatch(q, 10)
    idx.addUInt8Batch(more, np.arange(3000, 3500, dtype=np.int32))   # the graph no longer describes the data: rebuilt
    allrows = np.concatenate([data, more])
    set_ef(idx, 4096)
    h = idx.knnQueryBatch(q, 10)
    path = tmp_path / "appended.hnsw"
    idx.save(str(path))
    pi, pd, pc = port_answers(path, allrows, np.arange(3500, dtype=np.int32), q, 10, 4096, tmp_path)
    assert_knn_matches(h.ids, h.distances, h.sizes, pi, pd, pc, exact=True, what="appended rows, ef 4096")
    assert_same(*device_knn(idx, q, 10), h.ids, h.distances, "appended rows, device entry")
    with pytest.raises(nb.NmslibError) as e:                 # a query of the wrong length
        idx.knnQueryBatch(q[:, :64], 10)
    assert e.value.code == 9
    idx.deinit()

    small = nb.Index("l2sqr_sift", None, "hnsw", "DenseUInt8Vector", "Int")   # k above the row count
    small.addUInt8Batch(data[:40])
    small.buildIndex(nb.Params({"M": 8, "efConstruction": 40, "b200_build": "host"}))
    set_ef(small, 50)
    h = small.knnQueryBatch(q, 64)
    assert np.all(h.sizes == 40) and np.all(h.ids[:, 40:] == -1)
    path = tmp_path / "small.hnsw"
    small.save(str(path))
    pi, pd, pc = port_answers(path, data[:40], np.arange(40, dtype=np.int32), q, 64, 50, tmp_path)
    assert_knn_matches(h.ids, h.distances, h.sizes, pi, pd, pc, exact=True, what="k > n")
    assert_same(*device_knn(small, q, 64), h.ids, h.distances, "k > n, device entry")
    small.deinit()
