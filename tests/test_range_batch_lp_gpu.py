"""nmslib_b200_range_query_batch over l1 and linf: the exact CUDA-core scan (K2) in range mode, a fixed pass-1
threshold per query (linf: the radius; l1: the radius widened by the summation-order band), then the verification
kernel of the tensor-core range passes.  Every query gets exactly what nmslib_range_query_fill gives it: sizes, ids in
position order, distance bits, (float) radius."""
from types import SimpleNamespace

import numpy as np
import pytest

from nmslib_zig_b200 import synth
from oracle import oracle as O
from test_range_batch_gpu import ALL, assert_batch_is_single, make_index, spread

pytestmark = pytest.mark.gpu

LP = ["l1", "linf"]


def counters(idx):
    st = idx.stats()
    return st["range_tc_queries"], st["range_fallback_queries"], st["kernel_launches"]


def same_answers(a, b, what):
    assert np.array_equal(a.sizes, b.sizes), what
    assert np.array_equal(a.ids, b.ids), what
    assert np.array_equal(a.distances.view(np.int32), b.distances.view(np.int32)), what


def lp_radii(idx, q, n):
    """per query: 0; between the 10th and 11th neighbour; exactly a distance the single path reports (the boundary
    row must be in); 1e30; +inf.  Capacities 1, 25, 200 and n within one batch."""
    nq = len(q)
    k = min(n, 21)
    kd = idx.knnQueryBatch(q, k).distances.astype(np.float64)
    radii = np.empty(nq)
    for i in range(nq):
        kind = (i + n) % 5                               # (a batch of one query still sees every kind across n)
        if kind == 0:
            radii[i] = 0.0
        elif kind == 1:
            radii[i] = (kd[i, min(9, k - 1)] + kd[i, min(10, k - 1)]) / 2
        elif kind == 2:
            one = idx.rangeQuery(q[i], float(kd[i, k - 1]) * 1.01 + 1e-3, capacity=64)
            radii[i] = float(one.distances[len(one.distances) // 2])
        elif kind == 3:
            radii[i] = ALL
        else:
            radii[i] = np.inf
    caps = np.array([(1, 25, 200, n)[(i // 5 + i) % 4] for i in range(nq)])
    return radii, caps


@pytest.mark.parametrize("space", LP)
@pytest.mark.parametrize("dim", [1, 4, 31, 32, 33, 128, 129, 300, 768])
def test_dims(space, dim):
    n, nq = 20_011, 1_100
    data, q = synth.uniform(n, dim, 11) - 0.3, synth.uniform(nq, dim, 12) - 0.3
    idx = make_index(space, data)
    radii, caps = lp_radii(idx, q, n)
    tc0, _, _ = counters(idx)
    assert_batch_is_single(idx, q, radii, caps, spread(nq), f"{space}/{dim}")
    assert counters(idx)[0] == tc0                      # not a tensor-core pass
    idx.deinit()


@pytest.mark.parametrize("space", LP)
@pytest.mark.parametrize("n", [1, 127, 128, 129, 20_011])
@pytest.mark.parametrize("nq", [1, 127, 128, 129])
def test_row_and_query_counts(space, n, nq):
    """n around the 128-row tile, query counts around the 128-query CTA and the 256-query list block"""
    dim = 33
    data, q = synth.uniform(n, dim, 21) - 0.3, synth.uniform(nq, dim, 22) - 0.3
    idx = make_index(space, data)
    radii, caps = lp_radii(idx, q, n)
    assert_batch_is_single(idx, q, radii, caps, spread(nq), f"{space} n={n} nq={nq}")
    idx.deinit()


# ---------------------------------------------------------------- the l1 summation-order band
def seq_l1(data, q):
    """K2's pass-1 value: sum_i |q_i - x_i| added sequentially over the row, in float32"""
    acc = np.zeros(len(data), np.float32)
    for c in range(data.shape[1]):
        acc = acc + np.abs(q[c] - data[:, c])
    return acc


def lane_l1(data, q):
    """range_row_dist's value: lane l adds the float4 groups l, l + 32, ... (each group ((t0 + t1) + t2) + t3), then a
    butterfly over the 32 lanes, in float32 (zero padding to whole float4 groups changes no sum)"""
    n, dim = data.shape
    g = (dim + 3) // 4
    t = np.zeros((n, g * 4), np.float32)
    t[:, :dim] = np.abs(data - q[None, :])
    grp = ((t[:, 0::4] + t[:, 1::4]) + t[:, 2::4]) + t[:, 3::4]    # [n, g]
    lanes = np.zeros((n, 32), np.float32)
    for e in range(g):
        lanes[:, e % 32] = lanes[:, e % 32] + grp[:, e]
    for o in (16, 8, 4, 2, 1):
        lanes = lanes + lanes[:, np.arange(32) ^ o]
    return lanes[:, 0]


def test_l1_band_admits_rows_whose_sequential_sum_is_larger():
    """rows of a wide dynamic range: for many of them K2's sequential sum is strictly larger than the verified value.
    A query whose radius is exactly such a row's verified distance must get the row (a threshold T_q = r would drop
    it in pass 1), and one ulp below that radius must not."""
    rng = np.random.default_rng(5)
    n, dim, nq = 8_000, 200, 130
    mag = np.float32(2.0) ** rng.integers(-12, 12, size=(n, dim)).astype(np.float32)
    data = (rng.standard_normal((n, dim)).astype(np.float32) * mag).astype(np.float32)
    q = (rng.standard_normal((nq, dim)).astype(np.float32) * np.float32(0.01)).astype(np.float32)
    idx = make_index("l1", data)
    radii, rows = np.empty(nq), np.empty(nq, np.int64)
    for i in range(nq):
        s, v = seq_l1(data, q[i]), lane_l1(data, q[i])
        cand = np.nonzero(s > v)[0]
        assert len(cand) > 0
        j = cand[np.argmin(v[cand])]                     # the nearest such row: few rows lie within its distance
        rows[i], radii[i] = j, float(v[j])
    # the emulated verification value is the single path's distance, bit for bit
    for i in range(0, nq, 37):
        one = idx.rangeQuery(q[i], radii[i], capacity=n)
        hit = np.nonzero(one.ids == rows[i])[0]
        assert len(hit) == 1 and one.distances[hit[0]].view(np.int32) == np.float32(radii[i]).view(np.int32)
    r = assert_batch_is_single(idx, q, radii, np.full(nq, n), spread(nq), "l1 band")
    for i in range(nq):
        assert rows[i] in r.ids[i, :r.sizes[i]], f"query {i}: row {rows[i]} at the radius is missing"
    below = np.array([float(np.nextafter(np.float32(x), np.float32(-np.inf))) for x in radii])
    r = assert_batch_is_single(idx, q, below, np.full(nq, n), spread(nq), "l1 band, one ulp below")
    for i in range(nq):
        assert rows[i] not in r.ids[i, :r.sizes[i]]
    idx.deinit()


def test_linf_ties_at_the_radius():
    """many rows at exactly one linf distance from the query (exact arithmetic): the radius equal to it takes every one
    of them, one ulp below takes none"""
    rng = np.random.default_rng(7)
    dim, nq, per = 24, 130, 40
    q = rng.integers(-100, 100, size=(nq, dim)).astype(np.float32)
    d = np.float32(7.5)
    rows = []
    for i in range(nq):
        off = rng.integers(-29, 30, size=(per, dim)).astype(np.float32) * np.float32(0.25)   # |off| <= 7.25
        c = rng.integers(0, dim, size=per)
        off[np.arange(per), c] = np.where(rng.integers(0, 2, size=per) == 1, d, -d)
        rows.append(q[i] + off)
    far = rng.integers(-100, 100, size=(3_000, dim)).astype(np.float32) * np.float32(3.0)
    data = np.concatenate(rows + [far]).astype(np.float32)
    perm = rng.permutation(len(data))
    data = data[perm]
    idx = make_index("linf", data)
    n = len(data)
    at = assert_batch_is_single(idx, q, np.full(nq, 7.5), np.full(nq, n), spread(nq), "linf ties at r")
    below = float(np.nextafter(d, np.float32(0)))
    un = assert_batch_is_single(idx, q, np.full(nq, below), np.full(nq, n), spread(nq), "linf one ulp below")
    inv = np.argsort(perm)
    for i in range(nq):
        mine = inv[i * per:(i + 1) * per]                # positions of query i's tie rows
        got = set(at.ids[i, :at.sizes[i]].tolist())
        assert set(mine.tolist()) <= got
        assert np.all(at.distances[i, :at.sizes[i]] <= d)
        assert not set(mine.tolist()) & set(un.ids[i, :un.sizes[i]].tolist())
    idx.deinit()


@pytest.mark.parametrize("space", LP)
def test_inf_and_nan_elements(space):
    """rows holding +inf or NaN elements: l1 gives +inf / NaN, linf +inf / skips the NaN (fmaxf); radii +inf, NaN
    and finite ones"""
    n, dim, nq = 5_000, 40, 260
    data, q = synth.uniform(n, dim, 31) - 0.3, synth.uniform(nq, dim, 32) - 0.3
    data[::11, 3] = np.inf
    data[5::13, 7] = np.nan
    data[7::17, 0] = -np.inf
    idx = make_index(space, data)
    tenth = idx.knnQueryBatch(q, 10).distances[:, -1].astype(np.float64)
    for radius, what in ((np.full(nq, np.inf), "+inf"), (np.full(nq, np.nan), "NaN"), (tenth, "10th"),
                         (np.full(nq, ALL), "1e30")):
        for cap in (n, 30):
            r = assert_batch_is_single(idx, q, radius, np.full(nq, cap), spread(nq), f"{space} radius {what} cap {cap}")
            if what == "NaN":
                assert np.all(r.sizes == 0)
    idx.deinit()


@pytest.mark.parametrize("space", LP)
def test_cut_and_fallback(space):
    """a radius covering every row: with capacity n the lists overflow below the capacity and the queries are re-run
    per query (counted as fallbacks); with capacity 10 the position cut certifies them.  Neither counts as a
    tensor-core answer."""
    n, dim, nq = 100_000, 32, 300
    data, q = synth.uniform(n, dim, 41) - 0.3, synth.uniform(nq, dim, 42) - 0.3
    idx = make_index(space, data)
    tc0, fb0, _ = counters(idx)
    assert_batch_is_single(idx, q[:40], np.full(40, ALL), np.full(40, n), [0, 17, 39], f"{space} all rows, cap n")
    tc1, fb1, _ = counters(idx)
    assert fb1 > fb0 and tc1 == tc0
    assert_batch_is_single(idx, q, np.full(nq, ALL), np.full(nq, 10), spread(nq), f"{space} all rows, cap 10")
    tc2, fb2, _ = counters(idx)
    assert fb2 == fb1 and tc2 == tc0
    idx.deinit()


def test_one_pass_for_the_whole_batch():
    """1 100 certified l1 queries take a constant number of launches (scan + verification), not two per query"""
    n, dim, nq = 50_000, 64, 1_100
    data, q = synth.uniform(n, dim, 51) - 0.3, synth.uniform(nq, dim, 52) - 0.3
    idx = make_index("l1", data)
    tenth = idx.knnQueryBatch(q, 11).distances
    radii = ((tenth[:, 9].astype(np.float64) + tenth[:, 10]) / 2)
    tc0, fb0, l0 = counters(idx)
    r = idx.rangeQueryBatch(q, radii, 100)
    tc1, fb1, l1 = counters(idx)
    assert fb1 == fb0 and tc1 == tc0
    assert l1 - l0 <= 16, f"{l1 - l0} launches"
    assert np.all(r.sizes >= 10)
    assert_batch_is_single(idx, q, radii, np.full(nq, 100), spread(nq), "one pass")
    idx.deinit()


@pytest.mark.parametrize("space", LP)
def test_chunked_batch_equals_small_batches(space):
    """1 000 queries x capacity n of a 10 000-row index stage 80 MB of ids + distances: above the 64 MB budget of one
    chunk"""
    n, dim, nq = 10_000, 48, 1_000
    data, q = synth.uniform(n, dim, 61) - 0.3, synth.uniform(nq, dim, 62) - 0.3
    idx = make_index(space, data)
    radii = np.where(np.arange(nq) % 3 == 0, ALL, idx.knnQueryBatch(q, 31).distances[:, -1].astype(np.float64))
    big = idx.rangeQueryBatch(q, radii, n)
    for b in range(0, nq, 128):
        part = SimpleNamespace(ids=big.ids[b:b + 128], distances=big.distances[b:b + 128], sizes=big.sizes[b:b + 128])
        same_answers(idx.rangeQueryBatch(q[b:b + 128], radii[b:b + 128], n), part, f"{space} chunk {b}")
    idx.deinit()


@pytest.mark.parametrize("space", LP)
def test_appended_rows(space):
    n1, n2, dim, nq = 7_003, 3_333, 40, 300
    data, q = synth.uniform(n1 + n2, dim, 71) - 0.3, synth.uniform(nq, dim, 72) - 0.3
    ids = np.arange(n1 + n2, dtype=np.int32) * 2 + 5
    idx = make_index(space, data[:n1], ids=ids[:n1])
    radii, caps = lp_radii(idx, q, n1)
    assert_batch_is_single(idx, q, radii, caps, spread(nq), f"{space} before the append")
    idx.addDenseBatch(data[n1:], ids[n1:])
    radii, caps = lp_radii(idx, q, n1 + n2)
    assert_batch_is_single(idx, q, radii, caps, spread(nq), f"{space} after the append")
    idx.deinit()


@pytest.mark.parametrize("devices", ["0,0", "0,1"])
def test_linf_row_shards_answer_like_the_plain_index(devices):
    import torch
    if devices == "0,1" and torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    n, nq, dim = 12_345, 700, 24
    data, q = synth.uniform(n, dim, 81) - 0.3, synth.uniform(nq, dim, 82) - 0.3
    one = make_index("linf", data)
    grp = make_index("linf", data, {"b200_devices": devices})
    radii, caps = lp_radii(one, q, n)
    same_answers(one.rangeQueryBatch(q, radii, caps), grp.rangeQueryBatch(q, radii, caps), f"linf shards {devices}")
    one.deinit()
    grp.deinit()


@pytest.mark.parametrize("space", LP)
def test_against_the_oracle(space):
    """the ids within the radius are the oracle's (seq_knn over every row, filtered by <= float32(radius)), in
    position order"""
    n, dim = 6_000, 72
    data, q = synth.uniform(n, dim, 91) - 0.3, synth.uniform(5, dim, 92) - 0.3
    ids = np.arange(n, dtype=np.int32) * 3 + 7
    idx = make_index(space, data, ids=ids)
    oi, od, oc = O.seq_knn(space, data, q, n, ids)
    for want in (1, 57, 300):
        radius = np.array([(float(od[i][want - 1]) + float(od[i][want])) / 2 for i in range(len(q))])
        for cap in (400, 25):
            r = idx.rangeQueryBatch(q, radius, cap)
            for i in range(len(q)):
                inside = np.sort(oi[i][od[i] <= np.float32(radius[i])])
                assert np.array_equal(r.ids[i, :r.sizes[i]], inside[:cap]), f"{space} q{i} radius {radius[i]} cap {cap}"
    idx.deinit()


@pytest.mark.parametrize("space", LP)
def test_knn_unchanged_by_a_range_batch(space):
    n, dim, nq = 30_000, 128, 500
    data, q = synth.uniform(n, dim, 101) - 0.3, synth.uniform(nq, dim, 102) - 0.3
    idx = make_index(space, data)
    before = idx.knnQueryBatch(q, 20)
    radii, caps = lp_radii(idx, q, n)
    idx.rangeQueryBatch(q, radii, caps)
    after = idx.knnQueryBatch(q, 20)
    same_answers(before, after, f"{space} kNN before / after a range batch")
    idx.deinit()
