"""Bit-exact answers of every scan variant, on data whose arithmetic is exact.

uint8 rows are exact by construction; float rows of small integers are TF32-exact and keep every partial sum an integer
below 2^24.  On such data pass 1, the re-rank and the exact scan all produce exact distances, so a kNN answer has one
correct form: (distance, position) order, ids and distance bits equal to an int64 / float64 reference.  No tolerance,
and no swapping inside tie groups: ties resolve by insertion position (DESIGN.md, "Result order = one 64-bit key").

Covered: the uint8 norm digits at the top of their domain (max |x|^2 = 4 032 058 / 059 / 060 with zero rows), every
instantiation of the integer-pipe kernel (register list, buffer KPL 8 / 16, the dp4a scan for k > 256), the TF32 TS
kernel, pair kernel and single-CTA kernel on TF32-exact rows, the exact scan (K2) in all eight spaces through
force_exact=1, and the split (3xTF32) operands on rows of 32 floats (TS kernel) and 96 floats (pair kernel)."""
import math

import numpy as np
import pytest

import nmslib_zig_b200 as nb
from nmslib_zig_b200 import synth
from helpers import ATOL_COSINE, RTOL, assert_knn_matches, close, comparable
from oracle import oracle as O
from test_range_batch_gpu import make_index, spread
from test_range_batch_u8_gpu import boundary_rows, exact_d

pytestmark = pytest.mark.gpu

SP = "l2sqr_sift"
DEFAULTS = {"u8_imma": 1, "force_exact": 0, "tc_pair": 1, "tc_split": 1}
KS = [1, 12, 13, 40, 59, 60, 100, 256, 257]  # register list | buffer KPL 8 | buffer KPL 16 | exact scan (k > 256)


@pytest.fixture
def opts():
    """set process-wide options for one test; every option is back at its default afterwards"""
    def set_(**kw):
        for name, v in kw.items():
            nb.set_option(name, v)
    yield set_
    for name, v in DEFAULTS.items():
        nb.set_option(name, v)


def make_with(opts, space, data, params=None, **options):
    """an index created under `options` (force_exact and u8_imma are read when an index is created)"""
    opts(**options)
    try:
        return make_index(space, data, params)
    finally:
        opts(**{name: DEFAULTS[name] for name in options})


# ---------------------------------------------------------------------------------------------------- references
def ref_knn(D, k, fin=None):
    """exact kNN of distance matrix D [nq, n] (int64 or exact float64): per query the k smallest in (distance,
    position) order -- np.lexsort((position, distance)) -- as (ids [nq, k] padded with -1, float32 distances [nq, k]
    padded with +inf, sizes).  fin maps the selected D values to the reported float32 distance (l2: the fp32 root)."""
    nq, n = D.shape
    c = min(k, n)
    ids = np.full((nq, k), -1, np.int32)
    dist = np.full((nq, k), np.inf, np.float32)
    for i in range(nq):
        if c == 0:
            continue
        kth = np.partition(D[i], c - 1)[c - 1]
        cand = np.flatnonzero(D[i] <= kth)
        o = cand[np.lexsort((cand, D[i, cand]))][:c]
        ids[i, :c] = o
        dist[i, :c] = fin(D[i, o]) if fin else D[i, o].astype(np.float32)
    return ids, dist, np.full(nq, c, np.int64)


def ref_range(D_row, radius, cap):
    """the rows with d <= floor(radius) (uint8: the single-query conversion) in position order, truncated"""
    pos = np.flatnonzero(D_row <= math.floor(radius))[:cap]
    return pos.astype(np.int32), D_row[pos].astype(np.float32)


def assert_range_row(r, i, D_row, radius, cap, what):
    """row i of a range batch: the reference's size, ids and distance bits, then id -1 / +inf up to the width"""
    want_ids, want_d = ref_range(D_row, radius, cap)
    c = int(r.sizes[i])
    assert c == len(want_ids), f"{what}: query {i} size {c} != {len(want_ids)} (radius {radius!r})"
    assert np.array_equal(r.ids[i, :c], want_ids), f"{what}: query {i} ids differ (radius {radius!r})"
    assert np.array_equal(r.distances[i, :c].view(np.int32), want_d.view(np.int32)), f"{what}: query {i} distance bits"
    assert np.all(r.ids[i, c:] == -1) and np.all(np.isposinf(r.distances[i, c:])), f"{what}: query {i} padding"


def int_distances(space, X, Q):
    """exact distances [nq, n] of integer-valued rows as int64 (l2: the squared distance; the device orders l2 by it)"""
    x, q = np.asarray(X).astype(np.int64), np.asarray(Q).astype(np.int64)
    if space in ("l2", "l2sqr", SP):
        return (q * q).sum(1)[:, None] + (x * x).sum(1)[None, :] - 2 * q @ x.T
    if space == "negdotprod":
        return -(q @ x.T)
    out = np.empty((len(q), len(x)), np.int64)
    for i in range(len(q)):
        a = np.abs(x - q[i])
        out[i] = a.sum(1) if space == "l1" else a.max(1)
    return out


def fin_of(space):
    return (lambda d: np.sqrt(d.astype(np.float32))) if space == "l2" else None


def bits(d):
    """distance bits, -0.0 read as +0.0 (negdotprod reports -(q.x), so a zero product is -0.0 or +0.0 by formula)"""
    return (np.asarray(d, np.float32) + np.float32(0.0)).view(np.int32)


def assert_exact(r, want, what, rows=None):
    """ids, sizes and distance bits equal to the reference (rows: compare only those queries of r)"""
    ids, dist, sizes = want
    got_ids, got_d, got_s = (r.ids, r.distances, r.sizes) if rows is None else (r.ids[rows], r.distances[rows], r.sizes[rows])
    assert np.array_equal(got_s, sizes), f"{what}: sizes differ"
    bad = np.flatnonzero((got_ids != ids).any(1) | (bits(got_d) != bits(dist)).any(1))
    if bad.size:
        i = bad[0]
        j = int(np.flatnonzero((got_ids[i] != ids[i]) | (bits(got_d[i]) != bits(dist[i])))[0])
        raise AssertionError(f"{what}: {bad.size} of {len(ids)} queries differ; query {i if rows is None else rows[i]} "
                             f"rank {j}: got id {got_ids[i, j]} d {got_d[i, j]!r}, want id {ids[i, j]} d {dist[i, j]!r} "
                             f"(got {got_ids[i, :6].tolist()}, want {ids[i, :6].tolist()})")


def tie_bound_queries(D, k, gap):
    """queries whose k-th distance lies within `gap` - 1 of the (k + 4)-th: there the candidate lists (16 ranks in
    register mode, k + 6 survivors in buffer mode) may end inside the tie group and the certificate may fail.  Every
    other query must be certified by the tensor-core pass when its pass-1 error is below `gap` / 2."""
    n = D.shape[1]
    if n <= k + 3:
        return 0
    s = np.partition(D, (k - 1, k + 3), axis=1)
    return int(np.sum(s[:, k + 3] - s[:, k - 1] < gap))


def fallbacks(idx):
    return idx.stats()["fallback_queries"]


# ---------------------------------------------------------------------------------------------------- 1. uint8 digits
def norm_row(norm2):
    """a byte row of 128 with |x|^2 = norm2: 62 x 255, then the rest (4 032 058 / 059 / 060 are the domain's edge)"""
    tails = {4_032_058: [22, 4, 2, 2], 4_032_059: [22, 5], 4_032_060: [22, 5, 1]}
    row = np.zeros(128, np.uint8)
    row[:62] = 255
    row[62:62 + len(tails[norm2])] = tails[norm2]
    assert int((row.astype(np.int64) ** 2).sum()) == norm2
    return row


def small_norm_rows(rng, count, lo=1, hi=510):
    """`count` rows of 128 bytes with distinct |x|^2 in [lo, hi): one value a = isqrt(s) and s - a^2 ones"""
    out = np.zeros((count, 128), np.uint8)
    for r, s in enumerate(rng.choice(np.arange(lo, hi), size=count, replace=False)):
        a = math.isqrt(int(s))
        cols = rng.choice(128, size=1 + int(s) - a * a, replace=False)
        out[r, cols[0]] = a
        out[r, cols[1:]] = 1
    return out


def with_rows_at(base, specials):
    """base rows with specials {position: row} inserted so that each ends up at its position"""
    out = list(base)
    for pos in sorted(specials):
        out.insert(pos, specials[pos])
    return np.array(out, np.uint8)


def digit_data(top, layout):
    """sift-like rows + 150 rows with distinct |x|^2 < 510 + the row with |x|^2 = top + two all-zero rows.  With M at
    the top of the digit domain a zero row has the largest V(x) the digits must carry."""
    rng = np.random.default_rng(7)
    base = np.concatenate([synth.sift_like_u8(3_000, 101), small_norm_rows(rng, 150)])
    base = base[rng.permutation(len(base))]
    zero, edge = np.zeros(128, np.uint8), norm_row(top)
    where = {"fresh": {0: zero, 1_076: edge, 2_751: zero},     # zeros in the first and in a later tile and piece
             "same_shard": {0: zero, 900: zero, 1_200: edge},   # b200_devices=0,0: all in shard 0 (rows < 1 576)
             "split_shards": {0: zero, 900: zero, 2_500: edge}}[layout]
    return with_rows_at(base, where)


def digit_queries():
    rng = np.random.default_rng(8)
    return np.concatenate([np.zeros((1, 128), np.uint8), small_norm_rows(rng, 20), synth.sift_like_u8(20, 102)])


RADII = [0.0, 100.0, 508.5, 509.0, 510.0, 511.0, 1e30]


def check_digit_answers(idx, data, q, what):
    D = exact_d(data, q)
    for k in (1, 10, 40, 100):
        r = idx.knnQueryBatch(q, k)
        assert_exact(r, ref_knn(D, k), f"{what} k={k}")
    first_zero = np.flatnonzero(~data.any(1))[0]
    assert r.ids[0, 0] == first_zero and r.distances[0, 0] == 0.0, f"{what}: the zero query's nearest row is a zero row"
    cap = 400
    for radius in RADII:
        r = idx.rangeQueryBatch(q, radius, cap)
        assert r.ids.shape == (len(q), cap)
        for i in range(len(q)):
            assert_range_row(r, i, D[i], radius, cap, f"{what}: range batch")
        for i in (0, 1, 5, 30):
            one = idx.rangeQuery(q[i], radius, capacity=cap)
            want_ids, want_d = ref_range(D[i], radius, cap)
            assert np.array_equal(one.ids, want_ids), f"{what}: rangeQuery radius {radius} query {i}"
            assert np.array_equal(one.distances.view(np.int32), want_d.view(np.int32))


@pytest.mark.parametrize("top", [4_032_058, 4_032_059, 4_032_060])
def test_u8_digit_domain_edge(opts, top):
    """max |x|^2 at the edge of the digit domain: at 4 032 059 (M = 2 016 030) a zero row's V(x) = M needs d0 = 255;
    4 032 060 is one past the limit and takes the widened rows"""
    data, q = digit_data(top, "fresh"), digit_queries()
    idx = make_index(SP, data)
    check_digit_answers(idx, data, q, f"max |x|^2 {top}")
    assert idx.stats()["u8_imma"] == (0 if top > 4_032_059 else 1)
    idx.deinit()


@pytest.mark.parametrize("top", [4_032_058, 4_032_059, 4_032_060])
def test_u8_digit_domain_edge_arriving_in_an_append(opts, top):
    """the edge row and the zero rows are appended to an index already on the device: M and every row's digits are
    recomputed for the new maximum"""
    data, q = digit_data(top, "fresh"), digit_queries()
    special = [0, 1_076, 2_751]
    keep = np.setdiff1d(np.arange(len(data)), special)
    first, later = data[keep[:2_000]], np.concatenate([data[special[:1]], data[keep[2_000:2_600]], data[special[1:2]],
                                                       data[keep[2_600:]], data[special[2:]]])
    idx = make_index(SP, first)
    assert_exact(idx.knnQueryBatch(q, 10), ref_knn(exact_d(first, q), 10), "before the append")
    assert idx.stats()["u8_imma"] == 1
    full = np.concatenate([first, later])
    idx.addUInt8Batch(later, np.arange(len(first), len(full), dtype=np.int32))  # (ids = positions, as in `first`)
    check_digit_answers(idx, full, q, f"append, max |x|^2 {top}")
    assert idx.stats()["u8_imma"] == (0 if top > 4_032_059 else 1)
    idx.deinit()


@pytest.mark.parametrize("layout", ["same_shard", "split_shards"])
@pytest.mark.parametrize("top", [4_032_058, 4_032_059, 4_032_060])
def test_u8_digit_domain_edge_in_row_shards(opts, top, layout):
    """b200_devices=0,0: every shard takes M from its own rows -- the zero rows share a shard with the edge row
    (that shard's M is at the edge) or not"""
    data, q = digit_data(top, layout), digit_queries()
    idx = make_index(SP, data, {"b200_devices": "0,0"})
    check_digit_answers(idx, data, q, f"shards {layout}, max |x|^2 {top}")
    idx.deinit()


def test_u8_all_255_row_appended_to_byte_rows(opts):
    """appending an all-255 row (|x|^2 = 8 323 200, far past the digit block) switches an index on byte rows to the
    widened rows; the answers stay exact"""
    first = synth.sift_like_u8(5_000, 111)
    later = np.concatenate([synth.sift_like_u8(100, 112), np.full((1, 128), 255, np.uint8), synth.sift_like_u8(50, 113)])
    q = np.concatenate([synth.sift_like_u8(60, 114), np.full((1, 128), 255, np.uint8), np.zeros((1, 128), np.uint8)])
    idx = make_index(SP, first)
    assert_exact(idx.knnQueryBatch(q, 10), ref_knn(exact_d(first, q), 10), "byte rows")
    assert idx.stats()["u8_imma"] == 1
    full = np.concatenate([first, later])
    idx.addUInt8Batch(later, np.arange(len(first), len(full), dtype=np.int32))
    D = exact_d(full, q)
    for k in (1, 10, 100):
        assert_exact(idx.knnQueryBatch(q, k), ref_knn(D, k), f"widened k={k}")
    assert idx.stats()["u8_imma"] == 0
    r = idx.rangeQueryBatch(q, 150_000.5, 300)
    assert r.ids.shape == (len(q), 300)
    for i in range(len(q)):
        assert_range_row(r, i, D[i], 150_000.5, 300, "widened range batch")
    idx.deinit()


# ---------------------------------------------------------------------------------------------------- 2. uint8 kNN
def u8_planted(n, nq, seed):
    """sift-like rows and queries with duplicates across 64-row tiles and far-apart pieces, duplicate queries, and (for
    large n) groups of rows at one exact distance from a query: ties that only the position order resolves"""
    rng = np.random.default_rng(seed)
    data, q = synth.sift_like_u8(n, seed), synth.sift_like_u8(nq, seed + 1)
    if n > 1:
        data[-1] = data[0]
    for a in (63, 127, 255, n // 2):
        if a + 1 < n:
            data[a + 1] = data[a]
    q[0] = data[min(63, n - 1)]
    if nq > 2:
        q[-1] = data[0]
    if n >= 1_000 and nq >= 2:
        centres = rng.integers(20, 230, size=(2, 128)).astype(np.uint8)
        for qi, c in zip((1, nq // 2), centres):
            q[qi] = c
            group = boundary_rows(rng, c, 50, 24) + boundary_rows(rng, c, 51, 8)
            data[rng.choice(n, size=len(group), replace=False)] = np.array(group)
    return data, q


@pytest.mark.parametrize("n,nq", [(1, 1), (63, 255), (64, 256), (65, 257), (20_011, 1), (20_011, 1_100)])
def test_u8_knn_every_instantiation(opts, n, nq):
    """k = 1, 12 (register list), 13, 40, 59 (buffer, KPL 8), 60, 100, 256 (buffer, KPL 16), 257 (dp4a exact scan):
    the integer-pipe answer, the force_exact=1 answer and the int64 reference are identical"""
    data, q = u8_planted(n, nq, 17 + n % 7)
    D = exact_d(data, q)
    exact = make_with(opts, SP, data, force_exact=1)
    for k in KS:
        want = ref_knn(D, k)
        idx = make_index(SP, data)  # (a fresh index: certificate failures would widen the margin of later calls)
        assert_exact(idx.knnQueryBatch(q, k), want, f"u8 n={n} nq={nq} k={k}")
        if k <= 256:
            # pass 1 is exact up to +1 (the parity of |x|^2): where the k-th and (k+4)-th distances differ by 2 or more
            # the tensor-core pass must answer on its own
            assert fallbacks(idx) <= tie_bound_queries(D, k, 2), f"u8 n={n} nq={nq} k={k}: {fallbacks(idx)} fallbacks"
        assert idx.stats()["u8_imma"] == 1
        idx.deinit()
        assert_exact(exact.knnQueryBatch(q, k), want, f"u8 force_exact n={n} nq={nq} k={k}")
    exact.deinit()


# ---------------------------------------------------------------------------------------------------- 3. TF32-exact
FLOAT_SHAPES = {1: (63, 255), 4: (65, 257), 19: (1_601, 256), 32: (127, 513), 33: (129, 1), 100: (4_099, 300),
                128: (2_047, 257), 129: (257, 255), 160: (255, 256), 256: (513, 257), 768: (1_025, 300)}


def row_words(dim):
    return (dim + 31) // 32 * 32


SPARSE_NONZEROS = 32  # rows longer than 128 floats: nonzeros per row and query


def tf32_exact_max(dim):
    """largest value v such that rows of integers 0..v keep the certificate's bound E = row_words 2^-21 |q| max|x|
    below 0.4, with |q|, |x| <= v sqrt(m) for m values per row: all dim of them up to 128 floats (0..7 at 128), the
    SPARSE_NONZEROS of a sparse row beyond (1..12 at 160, 1..10 at 256, 1..5 at 768).  The tensor-core pass must then
    certify every query whose k-th distance is an integer below the (k + 4)-th.  (Dense rows of 0..3 at 256 or 0..1 at
    768 floats would tie at the k-th distance for most queries.)"""
    m = dim if dim <= 128 else SPARSE_NONZEROS
    return int(math.isqrt(int(0.4 * 2 ** 21 / (row_words(dim) * m))))


def tf32_exact_rows(rng, count, dim):
    v = tf32_exact_max(dim)
    if dim <= 128:
        return rng.integers(0, v + 1, size=(count, dim)).astype(np.float32)
    out = np.zeros((count, dim), np.float32)
    for r in range(count):
        out[r, rng.choice(dim, size=SPARSE_NONZEROS, replace=False)] = rng.integers(1, v + 1, size=SPARSE_NONZEROS)
    return out


def tf32_exact_data(dim, seed):
    n, nq = FLOAT_SHAPES[dim]
    rng = np.random.default_rng(seed)
    X, Q = tf32_exact_rows(rng, n, dim), tf32_exact_rows(rng, nq, dim)
    for a in (63, 255):
        if a + 1 < n:
            X[a + 1] = X[a]                       # a duplicate across a 64- / 256-row tile boundary
    Q[0] = X[n // 2]
    return X, Q


@pytest.mark.parametrize("dim", sorted(FLOAT_SHAPES))
def test_tf32_exact_rows_every_scan_variant(opts, dim):
    """l2sqr, l2 and negdotprod on the TS kernel (<= 128 floats) or the pair kernel (longer rows), at every k regime,
    bit-exact; rows longer than 128 floats also on the single-CTA kernel (tc_pair=0); force_exact=1 gives the same
    bits; l1 and linf (exact scan) too.  l2 is the fp32 root of an exact integer below 2^22, ordered by its square."""
    X, Q = tf32_exact_data(dim, dim)
    n, nq = len(X), len(Q)
    for space in ("l2sqr", "l2", "negdotprod"):
        D = int_distances(space, X, Q)
        exact = make_with(opts, space, X, force_exact=1)
        for k in KS:
            want = ref_knn(D, k, fin_of(space))
            what = f"{space}/{dim} n={n} nq={nq} k={k}"
            idx = make_index(space, X)
            assert_exact(idx.knnQueryBatch(Q, k), want, what)
            if k <= 256:
                assert fallbacks(idx) <= tie_bound_queries(D, k, 1), f"{what}: {fallbacks(idx)} fallbacks"
            if dim > 128 and k in (1, 13, 100):
                opts(tc_pair=0)
                assert_exact(idx.knnQueryBatch(Q, k), want, f"{what} tc_pair=0")
                opts(tc_pair=1)
            idx.deinit()
            assert_exact(exact.knnQueryBatch(Q, k), want, f"{what} force_exact")
        exact.deinit()
    sample = spread(nq)
    for space in ("l1", "linf"):
        D = int_distances(space, X, Q[sample])
        idx = make_index(space, X)
        for k in (1, 13, 100, 257):
            assert_exact(idx.knnQueryBatch(Q, k), ref_knn(D, k), f"{space}/{dim} k={k}", rows=sample)
        idx.deinit()


# ---------------------------------------------------------------------------------------------------- 4. exact scan
EXACT_SHAPES = [(1, 1), (127, 129), (129, 127), (5_000, 300)]


def float64_distances(space, X, Q, ids):
    """float64 distance of every (query, reported id) pair: cosinesimil 1 - nsp, angulardist acos(nsp)"""
    x, q = X.astype(np.float64)[np.maximum(ids, 0)], Q.astype(np.float64)[:, None, :]
    nsp = (x * q).sum(-1) / np.sqrt((x * x).sum(-1) * (q * q).sum(-1))
    nsp = np.clip(nsp, -1.0, 1.0)
    return 1.0 - nsp if space == "cosinesimil" else np.arccos(nsp)


@pytest.mark.parametrize("space", ["l2", "l2sqr", "negdotprod", "l1", "linf", SP, "cosinesimil", "angulardist"])
def test_exact_scan_all_spaces(opts, space):
    """K2 behind every failed certificate, selected for everything by force_exact=1: k = 1, 144 (shared-memory lists),
    145 (global lists), 300; exact spaces bit-exact, the cosine family against the oracle and a float64 distance"""
    rng = np.random.default_rng(5)
    for n, nq in EXACT_SHAPES:
        if space == SP:
            X, Q = synth.sift_like_u8(n, 41), synth.sift_like_u8(nq, 42)
        elif space in ("cosinesimil", "angulardist"):
            X, Q = synth.uniform(n, 40, 43) - 0.3, synth.uniform(nq, 40, 44) - 0.3
        else:
            X = rng.integers(0, 16, size=(n, 40)).astype(np.float32)
            Q = rng.integers(0, 16, size=(nq, 40)).astype(np.float32)
        idx = make_with(opts, space, X, force_exact=1)
        for k in (1, 144, 145, 300):
            r = idx.knnQueryBatch(Q, k)
            what = f"force_exact {space} n={n} nq={nq} k={k}"
            if space in ("cosinesimil", "angulardist"):
                oi, od, oc = O.seq_knn(space, X, Q, k)
                dist_of = lambda qi, i: O.pair_distance(space, X[i], Q[qi])
                assert_knn_matches(r.ids, comparable(space, r.distances), r.sizes, oi, comparable(space, od), oc,
                                   dist_of=lambda qi, i: comparable(space, dist_of(qi, i)), atol=ATOL_COSINE, what=what)
                c = min(k, n)
                d64 = float64_distances(space, X, Q, r.ids[:, :c])
                assert close(comparable(space, r.distances[:, :c]), comparable(space, d64), RTOL, ATOL_COSINE).all(), what
            else:
                assert_exact(r, ref_knn(int_distances(space, X, Q), k, fin_of(space)), what)
        idx.deinit()


# ---------------------------------------------------------------------------------------------------- 5. split operands
def dense_clusters(dim, delta, seed, nc=4, m=4_096, per=16):
    """nc clusters of m rows c + delta u (u ~ N(0, 1/dim) per value, rows not TF32-exact), shuffled, and `per` queries
    near each centre.  Every piece of the scan (a few hundred rows) then holds dozens of each cluster's rows, so every
    candidate list ends inside the query's cluster and the gap between the k-th and the (k + 6)-th pass-1 rank (a few
    1e-4 of |q| max|x|) lies inside the error band of TF32 operands (~2^-9 |q| max|x|) but outside that of split
    operands (~(D 2^-22 + 3 2^-20) |q| max|x|): the first certificate of every query fails and the engine re-runs the
    batch on split operands.  (Small clusters spread over many pieces do not do this: each piece then keeps the few
    members it holds, every list ends far outside the cluster, and the exact re-rank orders the near-duplicates.)"""
    rng = np.random.default_rng(seed)
    c = rng.random((nc, dim), dtype=np.float32)
    u = rng.normal(0, 1 / np.sqrt(dim), (nc, m, dim)).astype(np.float32)
    X = (c[:, None, :] + delta * u).reshape(-1, dim).astype(np.float32)
    Q = np.repeat(c, per, 0) + (0.01 * rng.normal(0, 1 / np.sqrt(dim), (nc * per, dim))).astype(np.float32)
    return X[rng.permutation(len(X))], Q.astype(np.float32)


@pytest.mark.parametrize("space,dim,delta", [("l2", 32, 0.3), ("negdotprod", 32, 0.02), ("l2", 96, 0.5)])
def test_split_operands(opts, space, dim, delta):
    """rows of <= 32 floats: the split rows (3 x 32 words) run on the TS kernel; 96 floats: 288 words, the pair kernel.
    The first batch fails its certificates and is re-run on split operands at once, the second starts there; both
    match the oracle, and the split pass certifies most queries (the rest go to the exact scan)"""
    X, Q = dense_clusters(dim, delta, dim)
    nq = len(Q)
    idx = make_index(space, X)
    for rep, k in enumerate((10, 40)):
        r = idx.knnQueryBatch(Q, k)
        st = idx.stats()
        oi, od, oc = O.seq_knn(space, X, Q, k)
        assert_knn_matches(r.ids, r.distances, r.sizes, oi, od, oc, what=f"split {space}/{dim} k={k}",
                           dist_of=lambda qi, i: O.pair_distance(space, X[i], Q[qi]))
        assert st["split_queries"] >= (rep + 1) * nq // 4, f"{space}/{dim} k={k}: split_queries {st['split_queries']}"
        assert st["fallback_queries"] <= (rep + 1) * nq // 4, \
            f"{space}/{dim} k={k}: {st['fallback_queries']} queries left for the exact scan after the split pass"
    idx.deinit()
