"""l2sqr_sift + hnsw saves and loads the reference's regular index file (Hnsw::SaveRegularIndexBin, hnsw.cc:810-842:
links only, the data set in the .dat next to it).  Host-side only: no device needed."""
from __future__ import annotations

import struct
from pathlib import Path

import numpy as np
import pytest

import nmslib_zig_b200 as nb
from nmslib_zig_b200 import synth
from oracle import oracle as O

GOLDEN = Path(__file__).resolve().parent / "golden"


def write_dat(path, data, ids):
    """Space::WriteObjectVectorBinData for uint8 rows: count, then per row buflen, id, label, datalen, bytes, sum x^2."""
    with open(str(path) + ".dat", "wb") as f:
        f.write(struct.pack("<Q", len(data)))
        for row, i in zip(np.asarray(data, np.uint8), np.asarray(ids, np.int32)):
            f.write(struct.pack("<QiiQ", 16 + 132, int(i), -1, 132))
            f.write(row.tobytes())
            f.write(struct.pack("<i", int(np.sum(row.astype(np.int64) ** 2))))


def load_u8(path, load_data=True):
    return nb.Index.load(str(path), "DenseUInt8Vector", "Int", load_data=load_data)


def host_built(n=600, seed=3):
    data = synth.sift_like_u8(n, seed)
    ids = (np.arange(n, dtype=np.int32) * 3 + 5)
    idx = nb.Index("l2sqr_sift", None, "hnsw", "DenseUInt8Vector", "Int")
    idx.addUInt8Batch(data, ids)
    idx.buildIndex(nb.Params({"M": 8, "efConstruction": 60, "b200_build": "host", "indexThreadQty": 1}))
    return idx, data, ids


def test_golden_regular_file_loads_and_saves_back_byte_identical(tmp_path):
    g = np.load(GOLDEN / "regular_hnsw_sift.npz")
    src = tmp_path / "golden.hnsw"
    src.write_bytes((GOLDEN / "regular_hnsw_sift.hnsw").read_bytes())
    write_dat(src, g["data"], g["ids"])
    idx = load_u8(src)
    assert idx.getSpaceType() == "l2sqr_sift" and idx.getMethod() == "hnsw"
    assert idx.getDataType() == "DenseUInt8Vector" and idx.dataQty() == len(g["data"])
    out = tmp_path / "again.hnsw"
    idx.save(str(out))
    assert out.read_bytes() == (GOLDEN / "regular_hnsw_sift.hnsw").read_bytes()
    assert Path(str(out) + ".dat").read_bytes() == Path(str(src) + ".dat").read_bytes()
    idx.deinit()


def test_host_built_index_round_trip(tmp_path):
    idx, data, ids = host_built()
    a = tmp_path / "a.hnsw"
    idx.save(str(a))
    idx.deinit()
    assert struct.unpack_from("<I", a.read_bytes(), 0)[0] == 0          # the regular format's flag
    one = load_u8(a)
    assert one.getSpaceType() == "l2sqr_sift" and one.getMethod() == "hnsw"
    assert one.getDataType() == "DenseUInt8Vector" and one.dataQty() == len(data)
    for pos in (0, 1, 299, len(data) - 1):
        assert np.array_equal(one.getDataPoint(pos), data[pos])
    b = tmp_path / "b.hnsw"
    one.save(str(b))
    one.deinit()
    assert a.read_bytes() == b.read_bytes()
    assert Path(str(a) + ".dat").read_bytes() == Path(str(b) + ".dat").read_bytes()


def test_saved_file_parses_with_the_independent_reader(tmp_path):
    """oracle.regular_to_flat_hnsw reads the regular layout on its own; the C port then searches the same graph.  On
    the golden graph the port answers the same from our re-saved file as from the reference's."""
    idx, data, ids = host_built()
    a = tmp_path / "a.hnsw"
    idx.save(str(a))
    idx.deinit()
    flat = O.regular_to_flat_hnsw(a, data, ids, tmp_path / "a.flat")
    port = O.PortHnsw(flat)
    assert port.total == len(data) and port.dim == 128
    q = synth.sift_like_u8(20, 4)
    pi, pd, pc, _ = port.knn(q.astype(np.float32), 5, 50)
    for i in range(len(q)):                       # every answer is an exact integer distance of a row of the data set
        for j in range(pc[i]):
            pos = int(np.nonzero(ids == pi[i, j])[0][0])
            assert pd[i, j] == O.pair_distance("l2sqr_sift", data[pos], q[i])
    port.close()

    g = np.load(GOLDEN / "regular_hnsw_sift.npz")
    src = tmp_path / "golden.hnsw"
    src.write_bytes((GOLDEN / "regular_hnsw_sift.hnsw").read_bytes())
    write_dat(src, g["data"], g["ids"])
    idx = load_u8(src)
    idx.save(str(tmp_path / "again.hnsw"))
    idx.deinit()
    qs = g["queries"].astype(np.float32)
    answers = []
    for path in (GOLDEN / "regular_hnsw_sift.hnsw", tmp_path / "again.hnsw"):
        p = O.PortHnsw(O.regular_to_flat_hnsw(path, g["data"], g["ids"], tmp_path / "x.flat"))
        answers.append(p.knn(qs, 10, 50)[:3])
        p.close()
    for x, y in zip(*answers):
        assert np.array_equal(x, y)


def test_load_failures_are_clean(tmp_path):
    idx, data, ids = host_built(n=300)
    a = tmp_path / "a.hnsw"
    idx.save(str(a))
    idx.deinit()
    with pytest.raises(nb.NmslibError) as e:                      # links only: the data set is required
        load_u8(a, load_data=False)
    assert e.value.code == 10
    bad = tmp_path / "bad.hnsw"                                   # a .dat with one row fewer than the graph has nodes
    bad.write_bytes(a.read_bytes())
    write_dat(bad, data[:-1], ids[:-1])
    with pytest.raises(nb.NmslibError):
        load_u8(bad)
    raw = a.read_bytes()                                          # a truncated links file
    for cut in (3, 20, len(raw) // 2, len(raw) - 1):
        t = tmp_path / f"t{cut}.hnsw"
        t.write_bytes(raw[:cut])
        write_dat(t, data, ids)
        with pytest.raises(nb.NmslibError):
            load_u8(t)
    nodat = tmp_path / "nodat.hnsw"                               # no .dat at all
    nodat.write_bytes(raw)
    with pytest.raises(nb.NmslibError) as e:
        load_u8(nodat)
    assert e.value.code == 10
    # every other combination behaves as before: a regular file loaded as float data is no float index
    with pytest.raises(nb.NmslibError):
        nb.Index.load(str(a))


@pytest.mark.skipif(not O.ref_available(), reason="oracle/_ref not built")
def test_reference_loads_our_regular_file(tmp_path):
    """The reference's own LoadIndex (Hnsw<int>, hnsw.cc) reads the file and answers like the C port on it."""
    idx, data, ids = host_built()
    a = tmp_path / "a.hnsw"
    idx.save(str(a))
    idx.deinit()
    q = synth.sift_like_u8(40, 4)
    ref = O.RefIndex("l2sqr_sift", "hnsw").add(data, ids).load(a)
    ref.set_query_params("efSearch=50")
    ri, rd, rc = ref.knn(q, 10)
    port = O.PortHnsw(O.regular_to_flat_hnsw(a, data, ids, tmp_path / "a.flat"))
    pi, pd, pc, _ = port.knn(q.astype(np.float32), 10, 50)
    assert np.array_equal(rc, pc) and np.array_equal(rd, pd)
    assert np.mean(ri == pi) >= 0.99                  # (the reference orders ties by heap address)
    ref.close()
    port.close()
