"""nmslib_b200_range_query_batch over uint8 indexes (l2sqr_sift) on the device.  Byte rows run the integer-pipe
kernel's range mode (an exact accumulator threshold per query), widened rows (option u8_imma=0, or norms beyond the
digit block) the TF32 pass; either way every query gets exactly what nmslib_range_query_fill gives it: sizes, ids in
position order, int distances bit for bit, radius floored."""
import numpy as np
import pytest

import nmslib_zig_b200 as nb
from nmslib_zig_b200 import synth
from helpers import assert_knn_matches
from oracle import oracle as O
from test_range_batch_gpu import ALL, assert_batch_is_single, make_index, mixed_radii, spread

pytestmark = pytest.mark.gpu

SP = "l2sqr_sift"


def make_u8(data, params=None, ids=None, **options):
    """a uint8 index created under process-wide options (read when an index is created), restored afterwards"""
    for k, v in options.items():
        nb.set_option(k, v)
    try:
        return make_index(SP, data, params, ids)
    finally:
        for k in options:
            nb.set_option(k, {"u8_imma": 1, "force_exact": 0}[k])


def exact_d(data, q):
    """int64 squared distances [nq, n] (the reference's int32 n1 + n2 - 2 x.y, exact)"""
    x, y = data.astype(np.int64), q.astype(np.int64)
    return (y * y).sum(1)[:, None] + (x * x).sum(1)[None, :] - 2 * y @ x.T


def counters(idx):
    st = idx.stats()
    return st["range_tc_queries"], st["range_fallback_queries"]


def same_answers(a, b):
    assert np.array_equal(a.sizes, b.sizes)
    assert np.array_equal(a.ids, b.ids)
    assert np.array_equal(a.distances.view(np.int32), b.distances.view(np.int32))


@pytest.mark.parametrize("nq", [1, 255, 257, 1_100])
def test_u8_batch_equals_single_bit_for_bit(nq):
    """20 011 rows (a ragged last tile); radii 0, half-integers, exactly a reported distance and 1e30; capacities
    1, 25, 200 and n in one batch.  Every query takes the integer-pipe pass; only a query whose radius covers every
    row with capacity n can need the per-query fallback (its lists overflow below the capacity)."""
    n = 20_011
    data, q = synth.sift_like_u8(n, 11), synth.sift_like_u8(nq, 12)
    idx = make_u8(data)
    radii, caps = mixed_radii(idx, SP, q, n)
    radii[1::4] = np.floor(radii[1::4]) + 0.5                # half-integers between the 10th and 11th neighbour
    tc0, fb0 = counters(idx)
    assert_batch_is_single(idx, q, radii, caps, spread(nq), f"u8 nq={nq}")
    tc1, fb1 = counters(idx)
    assert idx.stats()["u8_imma"] == 1
    assert (tc1 - tc0) + (fb1 - fb0) == nq
    assert fb1 - fb0 <= int(np.sum((radii == ALL) & (caps > 256)))
    # without that combination every query is answered by the tensor-core pass
    keep = ~((radii == ALL) & (caps > 256))
    if keep.any():
        assert_batch_is_single(idx, q[keep], radii[keep], caps[keep], spread(int(keep.sum())), f"u8 nq={nq} certified")
        tc2, fb2 = counters(idx)
        assert tc2 - tc1 == int(keep.sum()) and fb2 == fb1
    idx.deinit()


def boundary_rows(rng, q, d, count):
    """`count` rows at squared distance exactly d from q (sparse integer offsets, q + e stays within 0..255)"""
    rows = []
    dim = q.shape[0]
    while len(rows) < count:
        e = np.zeros(dim, np.int64)
        big = rng.choice(dim, size=rng.integers(0, 4), replace=False)
        e[big] = rng.integers(-5, 6, size=len(big))
        rest = d - int((e * e).sum())
        free = np.setdiff1d(np.arange(dim), big)
        if rest < 0 or rest > len(free):
            continue
        ones = rng.choice(free, size=rest, replace=False)
        e[ones] = rng.choice([-1, 1], size=rest)
        assert int((e * e).sum()) == d
        rows.append((q.astype(np.int64) + e).astype(np.uint8))
    return rows


def test_u8_parity_boundary():
    """the threshold is exact up to the parity of |x|^2: rows at exactly R come back, rows at R + 1 never do, for
    both parities of |x|^2 (|x|^2 = d - |q|^2 mod 2, so queries of both |q|^2 parities cover all four cases); radius
    R + 0.9 floors to R.  Also duplicates of a query (distance 0, radius 0) and all-zero query and database rows."""
    rng = np.random.default_rng(3)
    dim = 128
    qs = rng.integers(20, 230, size=(4, dim)).astype(np.uint8)
    norm2 = lambda v: int((v.astype(np.int64) ** 2).sum())
    if norm2(qs[0]) % 2 == norm2(qs[1]) % 2:                  # make the |q|^2 parities differ
        qs[1, 0] += 1
    qs[2] = 0                                                 # all-zero query
    qs[3] = qs[0]                                             # a repeated query
    special = []
    for i in (0, 1):
        for d in (49, 50, 51, 52, 53):
            special += boundary_rows(rng, qs[i], d, 6)
        special += [qs[i].copy() for _ in range(3)]         # duplicates: distance 0
    special += [np.zeros(dim, np.uint8) for _ in range(4)]
    filler = synth.sift_like_u8(6_000, 5)
    data = np.concatenate([filler, np.array(special)])
    data = data[rng.permutation(len(data))]                   # scattered over tiles and pieces
    idx = make_u8(data)
    D = exact_d(data, qs)
    for R in (0, 50, 51, 52):
        for radius in (float(R), R + 0.9):
            tc0, fb0 = counters(idx)
            r = assert_batch_is_single(idx, qs, np.full(len(qs), radius), np.full(len(qs), 400), range(len(qs)),
                                       f"parity R={R} radius={radius}")
            tc1, fb1 = counters(idx)
            assert tc1 - tc0 == len(qs) and fb1 == fb0
            for i in range(len(qs)):
                want = np.flatnonzero(D[i] <= R)
                got = r.ids[i, :r.sizes[i]]
                assert np.array_equal(got, want), f"q{i} R={R} radius={radius}"
                assert np.array_equal(r.distances[i, :r.sizes[i]], D[i, want].astype(np.float32))
                assert not np.any(D[i, got] == R + 1)
            if R >= 50:  # both sides of the boundary are populated, with both |x|^2 parities
                for i in (0, 1):
                    assert np.sum(D[i] == R) >= 6 and np.sum(D[i] == R + 1) >= 6
                par = {(int(D[i, j]), norm2(data[j]) % 2)
                       for i in (0, 1) for j in np.flatnonzero((D[i] == R) | (D[i] == R + 1))}
                assert {(R, 0), (R, 1), (R + 1, 0), (R + 1, 1)} <= par
    assert idx.stats()["u8_imma"] == 1
    idx.deinit()


def test_u8_against_the_oracle():
    """non-default ids: the ids within floor(radius) are the oracle's, in position order, int distances bit-exact"""
    n = 7_000
    data, q = synth.sift_like_u8(n, 21), synth.sift_like_u8(5, 22)
    ids = np.arange(n, dtype=np.int32) * 3 + 7
    idx = make_u8(data, ids=ids)
    oi, od, oc = O.seq_knn(SP, data, q, n, ids)
    for want in (1, 40, 300):
        for frac in (0.0, 0.5, 0.99):
            radius = np.array([float(od[i][want - 1]) + frac for i in range(len(q))])
            for cap in (500, 25):
                r = idx.rangeQueryBatch(q, radius, cap)
                for i in range(len(q)):
                    inside = od[i] <= np.floor(radius[i])
                    order = np.argsort(oi[i][inside])
                    exp_ids, exp_d = oi[i][inside][order][:cap], od[i][inside][order][:cap]
                    c = r.sizes[i]
                    assert np.array_equal(r.ids[i, :c], exp_ids), f"q{i} radius {radius[i]} cap {cap}"
                    assert np.array_equal(r.distances[i, :c].view(np.int32), exp_d.astype(np.float32).view(np.int32))
    idx.deinit()


def test_u8_position_cut_and_fallback():
    """a radius covering every row: with capacity 10 the position cut certifies every query; with capacity n some
    queries cannot be certified below the cut, re-run on the per-query scan, and still answer the same"""
    n, nq = 200_000, 2_000
    data, q = synth.sift_like_u8(n, 61), synth.sift_like_u8(nq, 62)
    idx = make_u8(data)
    tenth = idx.knnQueryBatch(q, 10).distances[:, -1].astype(np.float64)
    tc0, fb0 = counters(idx)
    assert_batch_is_single(idx, q, tenth, np.full(nq, 100), spread(nq, 24), "u8 typical")
    tc1, fb1 = counters(idx)
    assert tc1 - tc0 == nq and fb1 == fb0
    assert_batch_is_single(idx, q[:40], np.full(40, ALL), np.full(40, n), [0, 17, 39], "u8 all rows, capacity n")
    tc2, fb2 = counters(idx)
    assert fb2 - fb1 > 0
    assert_batch_is_single(idx, q, np.full(nq, ALL), np.full(nq, 10), spread(nq, 24), "u8 all rows, capacity 10")
    tc3, fb3 = counters(idx)
    assert fb3 == fb2 and tc3 - tc2 == nq
    idx.deinit()


def test_u8_widened_rows():
    """option u8_imma=0 and all-255 rows (norms beyond the digit block: widened on their own) run the TF32 pass; both
    answer like the single-query path, and u8_imma=0 answers exactly like the byte-row index over the same data"""
    n, nq = 20_011, 300
    data, q = synth.sift_like_u8(n, 31), synth.sift_like_u8(nq, 32)
    q[5] = 0
    q[6] = 255
    byte_rows = make_u8(data)
    widened = make_u8(data, u8_imma=0)
    radii, caps = mixed_radii(byte_rows, SP, q, n)
    assert byte_rows.stats()["u8_imma"] == 1 and widened.stats()["u8_imma"] == 0
    tc0, _ = counters(widened)
    a = assert_batch_is_single(widened, q, radii, caps, spread(nq), "u8_imma=0")
    assert counters(widened)[0] > tc0
    same_answers(a, byte_rows.rangeQueryBatch(q, radii, caps))
    byte_rows.deinit()
    widened.deinit()
    ext = np.concatenate([data[:9_000], np.full((8, 128), 255, np.uint8), data[9_000:12_000]])
    idx = make_u8(ext)
    radii, caps = mixed_radii(idx, SP, q, len(ext))
    radii[6] = 128 * 255 ** 2                                   # the all-255 query against the all-255 rows
    tc0, _ = counters(idx)
    assert_batch_is_single(idx, q, radii, caps, spread(nq), "all-255 rows")
    assert idx.stats()["u8_imma"] == 0
    assert counters(idx)[0] > tc0
    idx.deinit()


def test_u8_force_exact():
    """force_exact=1: the per-query exact scan for every query, same answers, no tensor-core pass counted"""
    n, nq = 20_011, 257
    data, q = synth.sift_like_u8(n, 41), synth.sift_like_u8(nq, 42)
    plain = make_u8(data)
    exact = make_u8(data, force_exact=1)
    radii, caps = mixed_radii(plain, SP, q, n)
    tc0, fb0 = counters(exact)
    a = assert_batch_is_single(exact, q, radii, caps, spread(nq, 16), "force_exact")
    assert counters(exact) == (tc0, fb0)
    same_answers(a, plain.rangeQueryBatch(q, radii, caps))
    plain.deinit()
    exact.deinit()


def test_u8_chunked_batch_equals_small_batches():
    """1 000 queries x capacity n of a 10 000-row index stage 80 MB of ids + distances: more than the 64 MB budget,
    so the batch runs in chunks"""
    n, nq = 10_000, 1_000
    data, q = synth.sift_like_u8(n, 71), synth.sift_like_u8(nq, 72)
    idx = make_u8(data)
    radii = np.where(np.arange(nq) % 3 == 0, ALL, idx.knnQueryBatch(q, 31).distances[:, -1].astype(np.float64))
    big = idx.rangeQueryBatch(q, radii, n)
    for b in range(0, nq, 128):
        part = idx.rangeQueryBatch(q[b:b + 128], radii[b:b + 128], n)
        assert np.array_equal(part.sizes, big.sizes[b:b + 128])
        assert np.array_equal(part.ids, big.ids[b:b + 128])
        assert np.array_equal(part.distances.view(np.int32), big.distances[b:b + 128].view(np.int32))
    idx.deinit()


@pytest.mark.parametrize("mixed", [False, True])
@pytest.mark.parametrize("devices", ["0,0", "0,1"])
def test_u8_row_shards_answer_like_the_plain_index(devices, mixed):
    """b200_devices: every shard runs the batch on its own rows; mixed = only the second shard holds all-255 rows, so
    the first runs on byte rows and the second on widened rows"""
    import torch
    if devices == "0,1" and torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    n, nq = 12_345, 700
    data, q = synth.sift_like_u8(n, 81), synth.sift_like_u8(nq, 82)
    if mixed:
        data[-5:] = 255
    one = make_u8(data)
    grp = make_u8(data, {"b200_devices": devices})
    radii, caps = mixed_radii(one, SP, q, n)
    tc0, fb0 = counters(grp)
    same_answers(one.rangeQueryBatch(q, radii, caps), grp.rangeQueryBatch(q, radii, caps))
    tc1, fb1 = counters(grp)
    assert (tc1 - tc0) + (fb1 - fb0) == 2 * nq                # (counted once per shard)
    one.deinit()
    grp.deinit()


def test_u8_knn_is_untouched_by_range_batches():
    """kNN, range batch, kNN on one index: both kNN answers are identical and match the oracle"""
    n, nq, k = 30_000, 600, 10
    data, q = synth.sift_like_u8(n, 91), synth.sift_like_u8(nq, 92)
    idx = make_u8(data)
    a = idx.knnQueryBatch(q, k)
    a_ids, a_d = a.ids.copy(), a.distances.copy()
    radii, caps = mixed_radii(idx, SP, q, n)
    idx.rangeQueryBatch(q, radii, caps)
    b = idx.knnQueryBatch(q, k)
    assert np.array_equal(a_ids, b.ids) and np.array_equal(a_d.view(np.int32), b.distances.view(np.int32))
    sample = spread(nq, 16)
    oi, od, oc = O.seq_knn(SP, data, q[sample], k)
    assert_knn_matches(b.ids[sample], b.distances[sample], b.sizes[sample], oi, od, oc, exact=True, what="u8 kNN")
    idx.deinit()
