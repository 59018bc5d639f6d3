"""The device HNSW build (csrc/hnsw_build_gpu.cu) link for link against its restatement (tests/hnsw_build_restate.py).

On rows whose every distance is an exact fp32 value, the build has one right answer: its candidate search is a
prefix kNN, heuristic 2 tests a strict <, the merge orders by (distance, id), the back-link sort is stable and no
two warps share a list.  The only freedom left is which of two keys of equal distance the scan returns at the K-th
place, and the data of every case is chosen so that no point depends on it (checked on the CPU by
test_hnsw_build_restate_cpu.py, and again here on the levels of the saved file).

Each case builds with b200_build=device, saves, and compares the file with the restatement: every level-0 and
upper-level list in order (the search expands lists in order), every count, maxlevel and the entry point, and the
build's batch and prune counts.

Not covered: the clamp of a batch to 32 768 new points, which needs more than 262 144 members on one level.
"""
import numpy as np
import pytest

import hnsw_build_restate as R
import nmslib_zig_b200 as nb

pytestmark = pytest.mark.gpu


def _first_diff(a, b):
    n = min(len(a), len(b))
    d = np.flatnonzero(np.asarray(a[:n]) != np.asarray(b[:n]))
    return int(d[0]) if d.size else n


@pytest.mark.parametrize("case", R.CASES, ids=lambda c: c.name)
def test_device_build_matches_restatement(case, tmp_path):
    X = R.case_rows(case)
    n = len(X)
    u8 = case.space == "l2sqr_sift"
    # external ids that are not the positions: the lists must hold positions all the same
    ids = (np.arange(n, dtype=np.int32)[::-1] * 3 + 1000) if case.ids else None
    idx = nb.Index(case.space, None, "hnsw", "DenseUInt8Vector" if u8 else "DenseVector", "Int" if u8 else "Float")
    (idx.addUInt8Batch if u8 else idx.addDenseBatch)(case.index_rows(X), ids)
    p = R.case_params(case)
    idx.buildIndex(nb.Params({**p, "b200_build": "device"}))
    idx.prepare()
    st = idx.stats()
    path = tmp_path / "g.hnsw"
    idx.save(str(path), False)
    idx.deinit()
    saved = R.read_regular(path) if u8 else R.read_optimized(path)
    if case.ids:
        assert np.array_equal(saved.ext_ids, ids)

    g = R.restated(case, saved.levels)
    assert not g.events.ambiguous, f"ambiguous points (level, batch, point): {g.events.ambiguous[:5]}"
    maxM = p.get("maxM", p["M"])
    assert (saved.maxM, saved.maxM0) == (maxM, p.get("maxM0", 2 * p["M"]))
    assert (saved.maxlevel, saved.enterpoint) == (g.maxlevel, g.enterpoint), "maxlevel / entry point"

    bad = [i for i in range(n)
           if saved.cnt0[i] != g.cnt0[i] or not np.array_equal(saved.links0[i], g.links0[i, :g.cnt0[i]])]
    if bad:
        i = bad[0]
        want = g.links0[i, :g.cnt0[i]].tolist()
        got = saved.links0[i].tolist()
        pytest.fail(f"{len(bad)} of {n} level-0 lists differ; node {i}: device {got}, restated {want} "
                    f"(first difference at {_first_diff(got, want)})")
    assert set(saved.upper) == set(g.upper), "upper-level membership"
    bad = [k for k in sorted(g.upper) if saved.upper[k] != g.upper[k]]
    if bad:
        k = bad[0]
        pytest.fail(f"{len(bad)} upper-level lists differ; node {k[0]} level {k[1]}: device {saved.upper[k]}, "
                    f"restated {g.upper[k]}")
    assert st["build_batches"] == g.batches, "batch count"
    assert st["build_prunes"] == g.prunes, "prune count"
