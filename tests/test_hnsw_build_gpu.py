"""Device-side HNSW construction (csrc/hnsw_build_gpu.cu, SURVEY 8f N3): prefix kNN on the tensor cores +
heuristic-2 selection + batched back links.  The graph is not the reference's graph (nor is the reference's
own from one run to the next), so the gate is recall parity: recall@10 at a given efSearch at or above what a
graph built by the host builder / by the reference itself reaches, plus the structural invariants of the
optimized-index layout (checked by searching the SAVED file with the oracle's port of the reference search)."""
from pathlib import Path

import numpy as np
import pytest

import nmslib_zig_b200 as nb
from helpers import recall
from nmslib_zig_b200 import synth
from oracle import oracle as O

pytestmark = pytest.mark.gpu
GOLDEN = Path(__file__).resolve().parent / "golden"


def _build(space, data, where, extra=None, dtype="DenseVector", dist="Float", ids=None):
    idx = nb.Index(space, None, "hnsw", dtype, dist)
    (idx.addUInt8Batch if dtype == "DenseUInt8Vector" else idx.addDenseBatch)(data, ids)
    p = {"M": 16, "efConstruction": 200, "b200_build": where}
    p.update(extra or {})
    idx.buildIndex(nb.Params(p))
    idx.prepare()
    return idx


def _sweep(idx, q, exact, efs=(20, 50, 100, 400)):
    out = []
    for ef in efs:
        idx.setQueryTimeParams(nb.Params({"efSearch": ef}))
        out.append(recall(idx.knnQueryBatch(q, 10).ids, exact))
    return out


@pytest.mark.parametrize("space,dim", [("l2", 48), ("cosinesimil", 200), ("negdotprod", 64)])
def test_device_built_graph_recall_vs_host_built(space, dim, tmp_path):
    n = 20_000
    if space == "negdotprod":
        data, q = synth.embedding_like(n, dim, 9), synth.embedding_like(300, dim, 10)
    else:
        data, q = synth.gist_like(n, dim, 41, clusters=16), synth.gist_like(300, dim, 42, clusters=16)
    exact, _, _ = O.seq_knn(space, data, q, 10)
    dev = _build(space, data, "device")
    st = dev.stats()
    assert st["build_total_ms"] > 0 and st["build_batches"] > 0, "the graph was not built on the device"
    host = _build(space, data, "host")
    assert host.stats()["build_total_ms"] == 0
    rd, rh = _sweep(dev, q, exact), _sweep(host, q, exact)
    for ef, a, b in zip((20, 50, 100, 400), rd, rh):
        assert a >= b - 0.015, f"{space} ef={ef}: device-built recall {a} < host-built {b}"
    assert rd[-1] >= 0.95
    # the saved file is a valid optimized index: the oracle's port of the reference search walks it to the same answers
    path = tmp_path / "dev.hnsw"
    dev.save(str(path), False)
    port = O.PortHnsw(path)
    pi, pd, pc, _ = port.knn(q, 10, 100)
    dev.setQueryTimeParams(nb.Params({"efSearch": 100}))
    r = dev.knnQueryBatch(q, 10)
    assert float(np.mean(r.ids == pi)) >= 0.99
    port.close()
    dev.deinit()
    host.deinit()


def test_device_built_graph_structure(tmp_path):
    """Link lists: within capacity, no self links, no duplicates, every id in range; every node but the first
    has at least one level-0 link; upper-level links stay inside their level."""
    import struct
    n, dim = 20_000, 32
    data = synth.gist_like(n, dim, 51, clusters=8)
    dev = _build("l2", data, "device", {"M": 12, "efConstruction": 100})
    path = tmp_path / "s.hnsw"
    dev.save(str(path), False)
    dev.deinit()
    g = nb.Index("l2", None, "hnsw")
    g.importHnsw(path)          # the reader validates the stream (sizes, offsets)
    raw = open(path, "rb").read()
    # header of Hnsw::SaveOptimizedIndex (hnsw.cc:774-806) as csrc/hnsw_format.cpp writes it: u32 version, u32 total,
    # u64 memoryPerObject, u64 offsetLevel0, u64 offsetData, i32 maxlevel, u32 enterpoint, u64 maxM, u64 maxM0,
    # i32 dist_func_type, u64 searchMethod
    _, total, mem_per, off_l0, _, maxlevel, enterpoint, maxM, maxM0, dist_func, _ = struct.unpack_from(
        "<IIQQQiIQQiQ", raw, 0)
    off = struct.calcsize("<IIQQQiIQQiQ")
    assert off == 68
    assert total == n and maxM == 12 and maxM0 == 24
    lvl0 = np.frombuffer(raw, np.uint8, total * mem_per, off).reshape(total, mem_per)
    cnt = lvl0[:, off_l0:off_l0 + 4].copy().view(np.int32)[:, 0]
    links = lvl0[:, off_l0 + 4:off_l0 + 4 + 4 * maxM0].copy().view(np.int32)
    assert cnt.max() <= maxM0 and cnt[1:].min() >= 1
    for i in range(0, n, 97):
        l = links[i, :cnt[i]]
        assert len(set(l.tolist())) == len(l) and i not in l and l.min() >= 0 and l.max() < n
    assert 0 <= enterpoint < n and maxlevel >= 2
    g.deinit()


def test_device_built_graph_recall_vs_reference_built(tmp_path):
    """The reference's graph is built here and now where oracle/_ref exists; elsewhere it is the one the reference built
    and saved as tests/golden/hnsw_l2_d32.hnsw (rows and ids regenerated as make_golden.py made them)."""
    if O.ref_available():
        n, dim = 30_000, 64
        data, q = synth.gist_like(n, dim, 5, clusters=32), synth.gist_like(400, dim, 6, clusters=32)
        ids, params = None, None
        ref = O.RefIndex("l2", "hnsw").add(data).build("M=16,efConstruction=200,indexThreadQty=8")
        path = tmp_path / "ref.hnsw"
        ref.save(path)
    else:
        data, q = synth.gist_like(2000, 32, 41, clusters=16), synth.gist_like(1000, 32, 43, clusters=16)
        ids, params = np.arange(2000, dtype=np.int32) + 1000, {"M": 8, "efConstruction": 100}
        path = GOLDEN / "hnsw_l2_d32.hnsw"
    exact, _, _ = O.seq_knn("l2", data, q, 10, ids)
    on_ref = nb.Index("l2", None, "hnsw")
    on_ref.importHnsw(path)
    assert np.array_equal(on_ref.getDataPoint(len(data) - 1), data[-1])
    dev = _build("l2", data, "device", params, ids=ids)
    r_ref, r_dev = _sweep(on_ref, q, exact), _sweep(dev, q, exact)
    for ef, a, b in zip((20, 50, 100, 400), r_dev, r_ref):
        assert a >= b - 0.01, f"ef={ef}: device-built recall {a} < reference-built {b}"
    on_ref.deinit()
    dev.deinit()


def test_device_build_uint8_rows():
    data, q = synth.sift_like_u8(20_000, 7), synth.sift_like_u8(200, 8)
    exact, _, _ = O.seq_knn("l2sqr_sift", data, q, 10)
    dev = _build("l2sqr_sift", data, "device", dtype="DenseUInt8Vector", dist="Int")
    assert dev.stats()["build_batches"] > 0
    dev.setQueryTimeParams(nb.Params({"efSearch": 400}))
    r = dev.knnQueryBatch(q, 10)
    assert recall(r.ids, exact) >= 0.95
    dev.deinit()


@pytest.mark.parametrize("n", [1, 3, 300, 2049])
def test_device_build_tiny_indexes(n):
    """Forced onto the device (b200_build=device) below the automatic threshold: single batch / single level /
    fewer rows than candidates asked for.  Every point must find itself, and on 300+ points recall must be ~1."""
    data = synth.gist_like(max(n, 1), 24, 61, clusters=4)[:n]
    dev = _build("l2", data, "device", {"M": 8, "efConstruction": 40})
    assert dev.stats()["build_total_ms"] > 0
    k = min(5, n)
    dev.setQueryTimeParams(nb.Params({"efSearch": 100}))
    r = dev.knnQueryBatch(data, k)
    assert np.all(r.sizes >= 1)
    if n >= 300:
        exact, _, _ = O.seq_knn("l2", data, data, k)
        assert recall(r.ids, exact) >= 0.99
        assert np.mean(r.ids[:, 0] == np.arange(n)) >= 0.99
    else:
        assert np.array_equal(r.ids[:, 0], np.arange(n))
    dev.deinit()
