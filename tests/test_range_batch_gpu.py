"""nmslib_b200_range_query_batch on the device: for every query the batch answers exactly what
nmslib_range_query_fill answers for it (sizes, ids in position order, distance bits), whichever path the
engine takes -- the tensor-core pass with verification, its position cut, the per-query exact fallback, the
exact per-query path of l1 / linf / l2sqr_sift, query chunks and row shards."""
import numpy as np
import pytest

import nmslib_zig_b200 as nb
from helpers import ATOL_COSINE, RTOL, comparable
from nmslib_zig_b200 import synth
from oracle import oracle as O

pytestmark = pytest.mark.gpu


def make_index(space, data, params=None, ids=None):
    u8 = space == "l2sqr_sift"
    idx = nb.Index(space, None, "seq_search", "DenseUInt8Vector" if u8 else "DenseVector", "Int" if u8 else "Float")
    (idx.addUInt8Batch if u8 else idx.addDenseBatch)(data, ids)
    idx.buildIndex(nb.Params(params) if params else None)
    return idx


def dataset(space, n, nq, dim, seed):
    if space == "l2sqr_sift":
        return synth.sift_like_u8(n, seed), synth.sift_like_u8(nq, seed + 1)
    return synth.uniform(n, dim, seed) - 0.3, synth.uniform(nq, dim, seed + 1) - 0.3


def spread(nq, m=40):
    """a spread sample: both ends of every 256-query block, the ragged tail, and evenly spaced queries"""
    s = {0, nq - 1}
    for b in range(0, nq, 256):
        s.update({b, min(nq - 1, b + 255)})
    s.update(np.linspace(0, nq - 1, m).astype(int).tolist())
    return sorted(s)


def assert_batch_is_single(idx, q, radii, caps, sample, what):
    r = idx.rangeQueryBatch(q, radii, caps)
    for i in sample:
        one = idx.rangeQuery(q[i], float(radii[i]), capacity=int(caps[i]))
        c = int(r.sizes[i])
        assert c == len(one.ids), f"{what}: query {i} size {c} != single {len(one.ids)} (radius {radii[i]!r})"
        assert np.array_equal(r.ids[i, :c], one.ids), f"{what}: query {i} ids differ"
        assert np.array_equal(r.distances[i, :c].view(np.int32), one.distances.view(np.int32)), \
            f"{what}: query {i} distance bits differ"
        assert np.all(r.ids[i, c:] == -1) and np.all(np.isinf(r.distances[i, c:]))
    return r


ALL = 1e30  # a radius larger than every distance


def mixed_radii(idx, space, q, n):
    """per query: 0, strictly between the 10th and 11th neighbour, exactly a distance the single path reports
    (the boundary row must be in), larger than every distance; capacities 1, 25, 200, n within one batch"""
    nq = len(q)
    kd = idx.knnQueryBatch(q, 21).distances.astype(np.float64)
    radii = np.empty(nq)
    for i in range(nq):
        kind = i % 4
        if kind == 0:
            radii[i] = 0.0
        elif kind == 1:
            radii[i] = max(0.0, (kd[i, 9] + kd[i, 10]) / 2)
        elif kind == 2:
            one = idx.rangeQuery(q[i], max(kd[i, 20], 0.0) * 1.01 + 1e-3, capacity=64)
            radii[i] = max(float(one.distances[len(one.distances) // 2]), 0.0) if len(one.distances) else 0.0
        else:
            radii[i] = ALL
    caps = np.array([(1, 25, 200, n)[(i // 4 + i) % 4] for i in range(nq)])
    return radii, caps


@pytest.mark.parametrize("space,dim", [("l2", 48), ("l2", 200), ("l2sqr", 128), ("l2sqr", 768),
                                       ("cosinesimil", 128), ("cosinesimil", 768), ("negdotprod", 48),
                                       ("negdotprod", 200), ("angulardist", 48), ("angulardist", 200),
                                       ("l1", 40), ("linf", 24), ("l2sqr_sift", 128)])
def test_batch_equals_single_bit_for_bit(space, dim):
    n, nq = 20_011, 1_100
    data, q = dataset(space, n, nq, dim, 11)
    idx = make_index(space, data)
    radii, caps = mixed_radii(idx, space, q, n)
    assert_batch_is_single(idx, q, radii, caps, spread(nq), f"{space}/{dim}")
    idx.deinit()


@pytest.mark.parametrize("space,dim", [("l2", 48), ("cosinesimil", 200)])
@pytest.mark.parametrize("nq", [1, 255, 257])
def test_query_counts(space, dim, nq):
    n = 9_001
    data, q = dataset(space, n, nq, dim, 21)
    idx = make_index(space, data)
    radii, caps = mixed_radii(idx, space, q, n)
    assert_batch_is_single(idx, q, radii, caps, spread(nq), f"{space}/{dim}/nq={nq}")
    idx.deinit()


@pytest.mark.parametrize("space,dim", [("l2", 48), ("cosinesimil", 200), ("negdotprod", 128), ("angulardist", 768)])
def test_against_the_oracle(space, dim):
    """the ids within the radius are the oracle's, in position order (tolerances of the single-query test)"""
    n = 6_000
    data, q = synth.uniform(n, dim, 1) - 0.3, synth.uniform(3, dim, 2) - 0.3
    ids = (np.arange(n, dtype=np.int32) * 3 + 7)
    idx = make_index(space, data, ids=ids)
    oi, od, oc = O.seq_knn(space, data, q, n, ids)
    for want in (1, 57, 300):
        radius = np.array([(float(od[i][want - 1]) + float(od[i][want])) / 2 for i in range(3)])
        if (radius < 0).any():
            continue
        for cap in (200, 25):
            r = idx.rangeQueryBatch(q, radius, cap)
            for i in range(3):
                ref_d = {int(a): float(b) for a, b in zip(oi[i], od[i])}
                inside = np.sort(oi[i][od[i] <= np.float32(radius[i])])
                got_ids = r.ids[i, :r.sizes[i]]
                assert np.array_equal(got_ids, inside[:cap]), f"{space} q{i} radius {radius[i]} cap {cap}"
                got = np.array([ref_d[int(a)] for a in got_ids], np.float32)
                assert np.allclose(comparable(space, r.distances[i, :r.sizes[i]]), comparable(space, got),
                                   rtol=RTOL * 4, atol=ATOL_COSINE)
    idx.deinit()


@pytest.mark.parametrize("space", ["cosinesimil", "angulardist"])
def test_zero_rows_and_zero_queries(space):
    n, dim = 5_000, 64
    data, q = dataset(space, n, 300, dim, 31)
    data[::7] = 0.0
    q[::5] = 0.0
    idx = make_index(space, data)
    for radius in (0.0, 0.5, 1.0, 1.0 + 1e-6, 1.7, 4.0):
        assert_batch_is_single(idx, q, np.full(len(q), radius), np.full(len(q), 300), spread(len(q)),
                               f"{space} zeros radius {radius}")
    idx.deinit()


def test_duplicate_rows_come_back_in_position_order():
    base = synth.uniform(500, 32, 41)
    data = np.repeat(base, 9, axis=0)                       # every row nine times
    q = base[:260] + 1e-3
    idx = make_index("l2", data)
    r = assert_batch_is_single(idx, q, np.full(len(q), 0.05), np.full(len(q), 40), spread(len(q)), "duplicates")
    for i in range(len(q)):
        got = r.ids[i, :r.sizes[i]]
        assert np.all(np.diff(got) > 0)                     # default ids are positions: strictly increasing
    idx.deinit()


@pytest.mark.parametrize("exact", [True, False])
def test_tf32_exact_and_inexact_data(exact):
    n, dim = 30_000, 96
    data, q = dataset("l2", n, 600, dim, 51)
    if exact:  # keep 10 mantissa bits: the rows and queries are TF32-exact, the error band is D 2^-22 only
        data = (data.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)
        q = (q.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)
    idx = make_index("l2", data)
    radii, caps = mixed_radii(idx, "l2", q, n)
    assert_batch_is_single(idx, q, radii, caps, spread(len(q)), f"tf32 exact={exact}")
    idx.deinit()


def test_paths_taken():
    n, dim, nq = 200_000, 128, 2_000
    data, q = dataset("l2", n, nq, dim, 61)
    idx = make_index("l2", data)
    tenth = idx.knnQueryBatch(q, 10).distances[:, -1].astype(np.float64)
    st0 = idx.stats()
    assert_batch_is_single(idx, q, tenth, np.full(nq, 100), spread(nq, 24), "typical")
    st = idx.stats()
    assert st["range_tc_queries"] - st0["range_tc_queries"] == nq
    assert st["range_fallback_queries"] - st0["range_fallback_queries"] == 0
    # a radius covering every row: with capacity n most queries cannot be certified below the position cut...
    small = q[:40]
    assert_batch_is_single(idx, small, np.full(40, ALL), np.full(40, n), [0, 17, 39], "all rows, capacity n")
    st2 = idx.stats()
    assert st2["range_fallback_queries"] - st["range_fallback_queries"] > 0
    # ...with capacity 10 the position cut certifies them
    assert_batch_is_single(idx, q, np.full(nq, ALL), np.full(nq, 10), spread(nq, 24), "all rows, capacity 10")
    st3 = idx.stats()
    assert st3["range_fallback_queries"] == st2["range_fallback_queries"]
    assert st3["range_tc_queries"] - st2["range_tc_queries"] == nq
    idx.deinit()


def test_chunked_batch_equals_small_batches():
    """1 000 queries x capacity n of a 10 000-row index stage 80 MB of ids + distances: more than the engine's
    64 MB budget, so the batch runs in chunks"""
    n, dim, nq = 10_000, 48, 1_000
    data, q = dataset("l2", n, nq, dim, 71)
    idx = make_index("l2", data)
    radii = np.where(np.arange(nq) % 3 == 0, ALL, idx.knnQueryBatch(q, 31).distances[:, -1].astype(np.float64))
    big = idx.rangeQueryBatch(q, radii, n)
    for b in range(0, nq, 128):
        part = idx.rangeQueryBatch(q[b:b + 128], radii[b:b + 128], n)
        assert np.array_equal(part.sizes, big.sizes[b:b + 128])
        assert np.array_equal(part.ids, big.ids[b:b + 128])
        assert np.array_equal(part.distances.view(np.int32), big.distances[b:b + 128].view(np.int32))
    idx.deinit()


@pytest.mark.parametrize("devices", ["0,0", "0,1"])
@pytest.mark.parametrize("space,dim", [("l2", 64), ("cosinesimil", 200), ("l1", 32)])
def test_row_shards_answer_like_the_plain_index(devices, space, dim):
    import torch
    if devices == "0,1" and torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    n, nq = 12_345, 700
    data, q = dataset(space, n, nq, dim, 81)
    one = make_index(space, data)
    grp = make_index(space, data, {"b200_devices": devices})
    radii, caps = mixed_radii(one, space, q, n)
    a, b = one.rangeQueryBatch(q, radii, caps), grp.rangeQueryBatch(q, radii, caps)
    assert np.array_equal(a.sizes, b.sizes)
    assert np.array_equal(a.ids, b.ids)
    assert np.array_equal(a.distances.view(np.int32), b.distances.view(np.int32))
    one.deinit()
    grp.deinit()


@pytest.mark.parametrize("dim", [200, 768])
def test_long_rows_without_the_pair_kernel(dim):
    """option tc_pair=0 (rows of more than 128 floats then have no range-mode kernel): the batch takes the per-query
    exact scan and still answers like the single-query path"""
    n, nq = 8_000, 300
    data, q = dataset("cosinesimil", n, nq, dim, 91)
    nb.set_option("tc_pair", 0)
    try:
        idx = make_index("cosinesimil", data)
        radii, caps = mixed_radii(idx, "cosinesimil", q, n)
        st0 = idx.stats()
        assert_batch_is_single(idx, q, radii, caps, spread(nq), f"tc_pair=0 cosinesimil/{dim}")
        assert idx.stats()["range_tc_queries"] == st0["range_tc_queries"]
        idx.deinit()
    finally:
        nb.set_option("tc_pair", 1)


@pytest.mark.parametrize("space", ["cosinesimil", "angulardist"])
def test_queries_of_tiny_norm(space):
    """|q|^2 below 2 FLT_MIN: the distance formula takes nsp = 0 (d = 1, or pi/2) for every row, whatever the pass-1
    ranks say -- every row must stay a candidate"""
    n, dim = 6_000, 64
    data, q = dataset(space, n, 260, dim, 95)
    q[::2] *= np.float32(1e-20)                     # |q|^2 ~ 1e-39
    idx = make_index(space, data)
    for radius in (1.0, 1.2, 1.5708, 2.5):
        r = assert_batch_is_single(idx, q, np.full(len(q), radius), np.full(len(q), 50), spread(len(q)),
                                   f"{space} tiny |q| radius {radius}")
        hit = 1.0 <= radius if space == "cosinesimil" else np.float32(np.pi / 2) <= np.float32(radius)
        if hit:
            assert np.all(r.sizes[::2] == 50)
    idx.deinit()
