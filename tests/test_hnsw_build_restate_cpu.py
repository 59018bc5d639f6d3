"""The restatement of the device HNSW build (tests/hnsw_build_restate.py) on hand-worked cases, and the data of
tests/test_hnsw_build_exact_gpu.py checked on the CPU: no point of any case is ambiguous (so the device graph has
one right answer), and the cases together exercise every rule of the build.  CPU only."""
import numpy as np

import hnsw_build_restate as R
import nmslib_zig_b200 as nb


def test_heuristic2_on_a_line():
    # base point 0 at x = 0; candidates x = 1, 2, -3, 5 at squared distances 1, 4, 9, 25
    sp = R.Space(0, [[0], [1], [2], [-3], [5]])
    cand, cd = np.array([[1, 2, 3, 4]]), np.array([[1, 4, 9, 25]])
    ev = R.Events()
    kid, kd, nk = R.heuristic2(sp, cand, cd, np.array([4]), 3, ev)
    # 1 is kept; 2 is 1 from kept 1 (< 4): dropped; -3 is 16 from 1 (>= 9): kept; 5 is 16 from 1 (< 25): dropped
    assert nk[0] == 2 and kid[0, :2].tolist() == [1, 3] and kd[0, :2].tolist() == [1, 9]
    assert ev.rejections == 2
    # fewer candidates than NN: all kept, in order, without a test
    kid, _, nk = R.heuristic2(sp, cand, cd, np.array([4]), 5, R.Events())
    assert nk[0] == 4 and kid[0, :4].tolist() == [1, 2, 3, 4]
    # NN reached: the walk stops
    kid, _, nk = R.heuristic2(sp, cand, cd, np.array([4]), 1, R.Events())
    assert nk[0] == 1 and kid[0, 0] == 1


def test_heuristic2_keeps_a_candidate_at_equal_distance():
    # base (0, 0); kept r = (2, 0) at 4; c = (1, 2) is 5 from the base and 1 + 4 = 5 from r: the test is strict
    sp = R.Space(0, [[0, 0], [2, 0], [1, 2]])
    kid, _, nk = R.heuristic2(sp, np.array([[1, 2]]), np.array([[4, 5]]), np.array([2]), 2, R.Events())
    assert nk[0] == 2 and kid[0].tolist() == [1, 2]


def test_batch_schedule():
    assert R.batches(1) == [] and R.batches(2) == [(0, 2)] and R.batches(256) == [(0, 256)]
    assert R.batches(257) == [(0, 256), (256, 257)]
    b = R.batches(4353)
    assert len(b) == 17 and b[15] == (3840, 4096) and b[16] == (4096, 4353)
    # a/8 rounded down to whole 256-point blocks, at least 256: 16 x 256 up to 4096, then 512, 768, 1024
    steps = [e - a for a, e in R.batches(10_000)]
    assert steps == [256] * 16 + [512] * 4 + [768] * 3 + [1024, 528]
    assert (R.efc_of(200), R.k_of(200)) == (200, 233)
    assert (R.efc_of(500), R.k_of(R.efc_of(500))) == (232, 256)
    assert (R.efc_of(1), R.k_of(1)) == (1, 9)


def test_ambiguity_check():
    # distances of the new point to positions 0..4; sorted: 1 (p1), 2 (p2), 3 (p3), 3 (p4), 5 (p0)
    d = [5, 1, 2, 3, 3]
    # K = 3: the 3rd and 4th distances tie.  i = 4: p1, p2 are closer and below i (2 < efc = 3), p3 ties and is
    # below i -- the scan may return p3 or p4, and the filter keeps p3 but drops p4
    assert R.is_ambiguous(d, 4, 3, 3)
    assert not R.is_ambiguous(d, 4, 3, 2)   # efc filled by p1, p2 before the tie
    assert not R.is_ambiguous(d, 2, 3, 3)   # both tied keys are at or behind i: dropped whichever is taken
    assert not R.is_ambiguous(d, 4, 5, 3)   # the scan returns all b <= K rows
    assert not R.is_ambiguous([5, 1, 2, 3, 4], 4, 3, 3)


def test_back_links_are_sorted_stably():
    # new points 10, 11, 12 (in this order) link to neighbour 3 at 7, 5, 7; 12 also links to 4
    runs = R.back_link_runs([10, 11, 12, 12], [3, 3, 3, 4], [7, 5, 7, 1])
    assert [(c, s.tolist(), d.tolist(), t) for c, s, d, t in runs] == [(3, [11, 10, 12], [5, 7, 7], 3),
                                                                      (4, [12], [1], 1)]
    # 40 new points at one distance: the first HB_MAXIN of them in their own order
    (c, s, d, t), = R.back_link_runs(np.arange(100, 140), np.zeros(40, int), np.full(40, 9))
    assert c == 0 and t == 40 and s.tolist() == list(range(100, 132))


def _host_levels(case, tmp_path):
    """Levels as the device build draws them (hnsw_assign_levels, shared with the host builder): a minimal host
    build with the case's M and mult, saved and read back."""
    n = len(R.case_rows(case))
    p = {"M": R.case_params(case)["M"], "efConstruction": 1, "b200_build": "host"}
    if "mult" in case.params:
        p["mult"] = case.params["mult"]
    idx = nb.Index("l2", None, "hnsw")
    idx.addDenseBatch(np.zeros((n, 4), np.float32) + np.arange(n, dtype=np.float32)[:, None])
    idx.buildIndex(nb.Params(p))
    path = tmp_path / f"{case.name}.hnsw"
    idx.save(str(path), False)
    idx.deinit()
    return R.read_optimized(path).levels


def test_exact_cases_are_unambiguous_and_cover_every_rule(tmp_path):
    total = R.Events()
    members = set()
    for case in R.CASES:
        levels = _host_levels(case, tmp_path)
        g = R.restated(case, levels)
        assert not g.events.ambiguous, f"{case.name}: ambiguous points (level, batch, point) {g.events.ambiguous[:5]}"
        total.add(g.events)
        members |= {int(np.count_nonzero(levels >= l)) for l in range(1, g.maxlevel + 1)}
        if case.name == "hub":
            assert g.events.long_runs > 0 and g.events.merge_ties > 0
    assert total.rejections > 0, "no heuristic-2 rejection"
    assert total.merges > 0, "no link step merged"
    assert total.merge_ties > 0, "no merged list with equal distances"
    assert total.long_runs > 0, f"no run longer than {R.HB_MAXIN}"
    assert total.short_filters > 0, "no prefix filter ended below efc"
    assert {2, 3} <= members, "no level of 2 and of 3 members"
