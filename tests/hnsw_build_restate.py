"""A restatement of the device HNSW build (csrc/hnsw_build_gpu.cu, DESIGN.md K6) for exact-arithmetic data.

It follows what the kernels do, not what the reference does: candidates are a prefix kNN over the batch schedule,
heuristic 2 keeps a candidate unless a kept neighbour is STRICTLY closer to it than the base point, back links are
sorted stably by (neighbour, distance) and each neighbour takes the first HB_MAXIN of its run, and a full list is
merged in (distance, id) order and re-pruned with heuristic 2 down to its capacity.

Rows are integer vectors and distances integers in int64 -- the graph distance in units the kernels compute exactly
in fp32 when every partial sum is an integer below 2^24:
  kind 0 (l2, l2sqr_sift)   squared l2 of the rows;
  kind 1 (cosinesimil)      rows are a / 4096 with sum(a^2) = 2^24 and a >= 0: 1 - dot = (2^24 - a.b) / 2^24,
                            so the unit here is 2^-24 and the distance is 2^24 - a.b (clamped as hb_finish does);
  kind 2 (negdotprod)       -a.b.
On such data the device graph is a function of the rows, the levels and the parameters, except where the scan may
return either of two keys of equal distance at the K-th place (`ambiguous`, see build_level()).
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

HB_MAXC = 256      # candidates per new point (hnsw_build_gpu.cu)
HB_MAXIN = 32      # back links a neighbour takes per batch
MAX_BATCH = 32768  # not reached here: it needs more than 262 144 points on a level
COS_ONE = 1 << 24  # kind 1: distance unit 2^-24

KIND = {"l2": 0, "l2sqr_sift": 0, "cosinesimil": 1, "negdotprod": 2}
_POS_BITS = 24     # key = (distance + offset) << _POS_BITS | position
_OFFSET = 1 << 30


def efc_of(ef_construction: int) -> int:
    """efConstruction as the device uses it: capped so that the slack fits the scan's largest k."""
    return min(ef_construction, HB_MAXC - 24)


def k_of(efc: int) -> int:
    """Keys the scan returns per new point."""
    return min(HB_MAXC, efc + efc // 8 + 8)


def batches(m: int) -> list[tuple[int, int]]:
    """The batch schedule [a, b) of a level of m members (none below 2 members)."""
    out: list[tuple[int, int]] = []
    if m < 2:
        return out
    a = 0
    while a < m:
        step = min(MAX_BATCH, max(256, a // 8 // 256 * 256))
        b = min(m, a + step)
        out.append((a, b))
        a = b
    return out


def is_ambiguous(dist_row, i: int, K: int, efc: int) -> bool:
    """dist_row: the distances of new point i to the members [0, b).  When the K-th and (K+1)-th smallest distances
    are equal, the scan may fill the places of that distance with any of the keys that have it.  The candidates can
    change only if the prefix filter reaches the first of those places (fewer than efc keys with a position below i
    are closer) and one of the tied keys has a position below i (otherwise the filter drops whichever is taken)."""
    d = np.asarray(dist_row, np.int64)
    b = d.shape[0]
    if b <= K:
        return False
    dk = np.partition(d, [K - 1, K])[K - 1:K + 1]
    if dk[0] != dk[1]:
        return False
    pos = np.arange(b)
    return int(np.count_nonzero((d < dk[0]) & (pos < i))) < efc and bool(np.any((d == dk[0]) & (pos < i)))


def back_link_runs(src, nbr, dist):
    """Back links (new point src[t] -> neighbour nbr[t] at distance dist[t]), listed in the order of the new points
    and, inside a point, of its kept list.  Returns [(neighbour, [sources], [distances], run length)] in neighbour
    order: a stable sort on (neighbour, distance), each neighbour keeping the first HB_MAXIN of its run."""
    src, nbr, dist = (np.asarray(x, np.int64) for x in (src, nbr, dist))
    order = np.lexsort((dist, nbr))  # (lexsort is stable: equal keys stay in the order of the new points)
    s, n, d = src[order], nbr[order], dist[order]
    out = []
    starts = np.flatnonzero(np.r_[True, n[1:] != n[:-1]]) if n.size else np.zeros(0, np.int64)
    ends = np.r_[starts[1:], n.size]
    for a, b in zip(starts, ends):
        e = min(b, a + HB_MAXIN)
        out.append((int(n[a]), s[a:e], d[a:e], int(b - a)))
    return out


class Space:
    """Integer rows of one level and the kernels' graph distance on them."""

    def __init__(self, kind: int, rows):
        self.kind = kind
        self.X = np.ascontiguousarray(rows, np.int64)
        self.Xf = self.X.astype(np.float64)
        self.sq = (self.X * self.X).sum(1)

    def _finish(self, dot):
        if self.kind == 1:
            return np.maximum(0, COS_ONE - np.clip(dot, -COS_ONE, COS_ONE))
        return -dot

    def block(self, a: int, b: int):
        """[b - a, b]: distances of the members [a, b) to the members [0, b)."""
        g = np.rint(self.Xf[a:b] @ self.Xf[:b].T).astype(np.int64)  # (float64 sums of integers below 2^53: exact)
        if self.kind == 0:
            return self.sq[a:b, None] + self.sq[None, :b] - 2 * g
        return self._finish(g)

    def pair(self, u, v):
        """Element-wise distances of members u and v (broadcast)."""
        if self.kind == 0:
            diff = self.X[u] - self.X[v]
            return (diff * diff).sum(-1)
        return self._finish((self.X[u] * self.X[v]).sum(-1))


@dataclass
class Events:
    """What the restated build went through (so a test can show that no rule was exercised by luck only)."""
    rejections: int = 0        # heuristic 2 dropped a candidate
    merges: int = 0            # a link step took the merge path
    merge_ties: int = 0        # a merged list held two links of equal distance (ordered by id)
    long_runs: int = 0         # a neighbour had more than HB_MAXIN incoming links in one batch
    short_filters: int = 0     # the prefix filter ended below efc although the scan had more than K rows
    ambiguous: list = field(default_factory=list)  # (level, batch start, local index) of ambiguous points

    def add(self, o: "Events"):
        self.rejections += o.rejections
        self.merges += o.merges
        self.merge_ties += o.merge_ties
        self.long_runs += o.long_runs
        self.short_filters += o.short_filters
        self.ambiguous += o.ambiguous


def heuristic2(sp: Space, cand, cd, m, NN: int, ev: Events):
    """hb_heuristic2 for many base points at once.  cand / cd: [r, W] candidates by increasing distance to base
    (valid where column < m).  Fewer than NN candidates are all kept; otherwise a candidate c is kept unless some
    kept r has d(c, r) < d(c, base), until NN are kept.  Returns kept ids [r, NN], distances [r, NN], counts [r]."""
    r, W = cand.shape
    kid = np.full((r, NN), -1, np.int64)
    kd = np.zeros((r, NN), np.int64)
    nk = np.zeros(r, np.int64)
    small = m < NN
    if small.any():
        w = min(W, NN)
        cols = np.arange(w)[None, :] < m[small, None]
        kid[small, :w] = np.where(cols, cand[small, :w], -1)
        kd[small, :w] = np.where(cols, cd[small, :w], 0)
        nk[small] = m[small]
    walk = ~small
    for j in range(W):
        act = np.flatnonzero(walk & (j < m) & (nk < NN))
        if act.size == 0:
            break
        c, dc = cand[act, j], cd[act, j]
        kmax = int(nk[act].max())
        good = np.ones(act.size, bool)
        if kmax:
            valid = np.arange(kmax)[None, :] < nk[act, None]
            kept = np.where(valid, kid[act, :kmax], 0)
            closer = valid & (sp.pair(c[:, None], kept) < dc[:, None])
            good = ~closer.any(1)
        ev.rejections += int(act.size - good.sum())
        at = act[good]
        kid[at, nk[at]] = c[good]
        kd[at, nk[at]] = dc[good]
        nk[at] += 1
    return kid, kd, nk


def build_level(sp: Space, m: int, cap: int, M: int, ef_construction: int, level: int = 0):
    """One level over its m members (local index = insertion order).  Returns links [m, cap] (-1 unused),
    counts [m], batch count, prune count, events."""
    links = np.full((m, cap), -1, np.int64)
    ldist = np.zeros((m, cap), np.int64)
    cnt = np.zeros(m, np.int64)
    ev = Events()
    Ml = min(M, cap)
    efc = efc_of(ef_construction)
    K = k_of(efc)
    prunes = 0
    sched = batches(m)
    for a, b in sched:
        nq = b - a
        D = sp.block(a, b)
        pos = np.arange(b, dtype=np.int64)
        keys = ((D + _OFFSET) << _POS_BITS) | pos[None, :]
        if b > K:
            part = np.partition(keys, [K - 1, K], axis=1)
            kplus = part[:, K] >> _POS_BITS
            keys = np.sort(part[:, :K], axis=1)
        else:
            kplus = None
            keys = np.sort(keys, axis=1)
        kpos = keys & ((1 << _POS_BITS) - 1)
        kdist = (keys >> _POS_BITS) - _OFFSET
        me = np.arange(a, b, dtype=np.int64)[:, None]
        ok = kpos < me
        rank = np.cumsum(ok, axis=1)
        take = ok & (rank <= efc)
        mq = np.minimum(rank[:, -1], efc)
        if kplus is not None:
            ev.short_filters += int(np.count_nonzero(mq < efc))
            dk = keys[:, K - 1] >> _POS_BITS
            for w in np.flatnonzero(dk == kplus):  # (is_ambiguous on the few rows whose K-th distance is tied)
                if is_ambiguous(D[w], a + w, K, efc):
                    ev.ambiguous.append((level, a, a + int(w)))
        W = max(1, int(mq.max()))
        cand = np.full((nq, W), -1, np.int64)
        cd = np.zeros((nq, W), np.int64)
        rw, cl = np.nonzero(take)
        col = rank[rw, cl] - 1
        cand[rw, col] = kpos[rw, cl]
        cd[rw, col] = kdist[rw, cl]
        kid, kd, nk = heuristic2(sp, cand, cd, mq, Ml, ev)
        # select: the forward lists of the new points
        links[a:b, :Ml] = np.where(np.arange(Ml)[None, :] < nk[:, None], kid, -1)
        ldist[a:b, :Ml] = kd
        cnt[a:b] = nk
        # back links, then one link step per touched neighbour on the lists the select step left
        on = np.arange(Ml)[None, :] < nk[:, None]
        src = np.broadcast_to(me, (nq, Ml))[on]
        runs = back_link_runs(src, kid[on], kd[on])
        merge = []
        for c, s, d, total in runs:
            if total > HB_MAXIN:
                ev.long_runs += 1
            have, inc = int(cnt[c]), len(s)
            if have + inc <= cap:
                links[c, have:have + inc] = s
                ldist[c, have:have + inc] = d
                cnt[c] = have + inc
            else:
                merge.append((c, np.r_[links[c, :have], s], np.r_[ldist[c, :have], d]))
        if merge:
            Wm = max(len(x[1]) for x in merge)
            base = np.array([x[0] for x in merge], np.int64)
            mids = np.full((len(merge), Wm), -1, np.int64)
            mds = np.zeros((len(merge), Wm), np.int64)
            mm = np.zeros(len(merge), np.int64)
            for r, (c, ids, ds) in enumerate(merge):
                o = np.lexsort((ids, ds))  # (distance, id)
                mids[r, :len(ids)] = ids[o]
                mds[r, :len(ids)] = ds[o]
                mm[r] = len(ids)
                if np.any(np.diff(ds[o]) == 0):
                    ev.merge_ties += 1
            kid2, kd2, nk2 = heuristic2(sp, mids, mds, mm, cap, ev)
            links[base] = np.where(np.arange(cap)[None, :] < nk2[:, None], kid2, -1)
            ldist[base] = kd2
            cnt[base] = nk2
            ev.merges += len(merge)
            prunes += len(merge)
    return links, cnt, len(sched), prunes, ev


@dataclass
class Graph:
    links0: np.ndarray           # [n, maxM0] positions, -1 unused
    cnt0: np.ndarray             # [n]
    upper: dict                  # (position, level) -> list of positions
    maxlevel: int
    enterpoint: int
    batches: int
    prunes: int
    events: Events


def restate(space: str, rows, levels, M: int = 16, ef_construction: int = 200, maxM: int | None = None,
            maxM0: int | None = None) -> Graph:
    """The device build over integer rows with the given per-position levels (as the saved file records them)."""
    maxM = M if maxM is None else maxM
    maxM0 = 2 * M if maxM0 is None else maxM0
    levels = np.asarray(levels, np.int64)
    n = len(levels)
    maxlevel = int(levels.max())
    enterpoint = int(np.argmax(levels == maxlevel))  # the first position that reaches the top level
    kind = KIND[space]
    ev = Events()
    links0, cnt0, nb, npr, e = build_level(Space(kind, rows), n, maxM0, M, ef_construction, 0)
    ev.add(e)
    upper = {}
    for l in range(1, maxlevel + 1):
        mem = np.flatnonzero(levels >= l)
        lk, lc, b, p, e = build_level(Space(kind, np.asarray(rows)[mem]), len(mem), maxM, M, ef_construction, l)
        nb += b
        npr += p
        ev.add(e)
        for li, g in enumerate(mem):
            upper[(int(g), l)] = mem[lk[li, :lc[li]]].tolist()
    return Graph(links0, cnt0, upper, maxlevel, enterpoint, nb, npr, ev)


# ---- data on which every distance the build computes is an exact fp32 value ------------------------------------

def _rng(seed: int) -> np.random.Generator:
    return np.random.Generator(np.random.Philox(key=seed))


def l2_rows(n: int, dim: int, seed: int, clusters: int = 16, spread: int = 60, by_cluster: bool = False):
    """Integer rows in clusters, values in [0, 400]: squared distances and norms stay below 2^24 at dim <= 32.
    by_cluster: the rows come cluster after cluster, so the new points of a batch crowd each other's candidates."""
    rng = _rng(seed)
    cent = rng.integers(spread, 400 - spread, size=(clusters, dim))
    which = np.sort(rng.integers(0, clusters, n)) if by_cluster else rng.integers(0, clusters, n)
    return cent[which] + rng.integers(-spread, spread + 1, size=(n, dim))


def negdot_rows(n: int, dim: int, seed: int):
    """Signed integers in [-800, 800] (TF32-exact); at dim 20 every dot product stays below 2^24 in magnitude."""
    return _rng(seed).integers(-800, 801, size=(n, dim))


def cos_rows(n: int, dim: int, seed: int):
    """Integer vectors a with sum(a^2) = 2^24 and 0 <= a_i < 2048; the index gets a / 4096, unit rows whose
    components are TF32-exact and whose dot products are multiples of 2^-24 in [0, 1].  dim - 4 components are
    drawn, the rest of 2^24 is written as a sum of four squares."""
    rng = _rng(seed)
    out = np.zeros((n, dim), np.int64)
    sq = np.arange(2048, dtype=np.int64) ** 2
    for r in range(n):
        while True:
            head = rng.integers(0, 1100, dim - 4)
            rest = COS_ONE - int((head * head).sum())
            if rest < 0:
                continue
            a0, a1 = rng.integers(0, 2048, 2)
            rest2 = rest - a0 * a0 - a1 * a1
            if rest2 < 0:
                continue
            a2 = sq[sq <= rest2]
            r3 = rest2 - a2
            a3 = np.rint(np.sqrt(r3)).astype(np.int64)
            hit = np.flatnonzero((a3 * a3 == r3) & (a3 < 2048))
            if hit.size:
                h = hit[rng.integers(0, hit.size)]
                out[r] = np.r_[head, a0, a1, h, a3[h]]
                break
    assert np.all((out * out).sum(1) == COS_ONE)
    return out


def hub_rows(n: int, dim: int, seed: int):
    """A centre row at position 0 and points on a sphere around it (signed permutations of one integer vector):
    the centre is the nearest earlier point of most of them, far more than HB_MAXIN of one batch, all at the
    same distance."""
    rng = _rng(seed)
    base = rng.integers(20, 120, dim)
    centre = np.full(dim, 150)
    pts = np.stack([rng.permutation(base) * rng.choice([-1, 1], dim) for _ in range(n - 1)])
    return np.vstack([centre, centre + pts])


@dataclass
class Case:
    name: str
    space: str
    make: object        # seed -> integer rows
    seed: int
    params: dict
    ids: bool = False   # external ids that are not the positions

    def rows(self):
        return self.make(self.seed)

    def index_rows(self, X):
        if self.space == "cosinesimil":
            return (X / 4096.0).astype(np.float32)
        if self.space == "l2sqr_sift":
            return X.astype(np.uint8)
        return X.astype(np.float32)


def _sift(n, seed):
    from nmslib_zig_b200 import synth
    return synth.sift_like_u8(n, seed).astype(np.int64)


CASES = [
    Case("l2_d32", "l2", lambda s: l2_rows(10_000, 32, s), 311, {}, ids=True),
    Case("l2_d24", "l2", lambda s: l2_rows(6_000, 24, s), 312, {}),
    Case("negdot_d20", "negdotprod", lambda s: negdot_rows(6_000, 20, s), 113, {}),
    Case("cos_d24", "cosinesimil", lambda s: cos_rows(6_000, 24, s), 14, {}),
    Case("sift_u8", "l2sqr_sift", lambda s: _sift(5_000, s), 2915, {}),
    Case("prune_m2", "l2", lambda s: l2_rows(4_353, 24, s), 216, {"M": 2, "maxM0": 3}),
    Case("prune_m4", "negdotprod", lambda s: negdot_rows(4_000, 20, s), 17, {"M": 4, "maxM0": 4}),
    Case("m32", "l2", lambda s: l2_rows(3_000, 32, s), 118, {"M": 32}),
    Case("m64", "cosinesimil", lambda s: cos_rows(3_000, 24, s), 19, {"M": 64, "maxM0": 64}),
    Case("maxm_below_m", "l2", lambda s: l2_rows(4_000, 24, s), 620, {"M": 16, "maxM": 5, "mult": 0.8}),
    Case("efc1", "l2", lambda s: l2_rows(3_000, 24, s), 21, {"efConstruction": 1}),
    Case("efc500", "l2", lambda s: l2_rows(3_000, 32, s), 222, {"efConstruction": 500}),
    Case("crowded_batches", "l2", lambda s: l2_rows(5_000, 32, s, spread=100, by_cluster=True), 23, {"M": 8, "efConstruction": 40}),
    Case("many_levels", "l2", lambda s: l2_rows(2_000, 24, s), 1124, {"M": 6, "mult": 2.2}),
    Case("n2", "l2", lambda s: l2_rows(2, 24, s), 25, {}),
    Case("n3", "l2", lambda s: l2_rows(3, 24, s), 26, {}),
    Case("n255", "l2", lambda s: l2_rows(255, 24, s), 27, {}),
    Case("n256", "l2", lambda s: l2_rows(256, 24, s), 28, {}),
    Case("n257", "l2", lambda s: l2_rows(257, 24, s), 29, {}),
    Case("hub", "l2", lambda s: hub_rows(2_000, 24, s), 130, {"M": 8, "efConstruction": 60}),
]


# ---- the saved graph -------------------------------------------------------------------------------------------

@dataclass
class Saved:
    maxlevel: int
    enterpoint: int
    maxM: int
    maxM0: int
    levels: np.ndarray   # [n]
    cnt0: np.ndarray     # [n]
    links0: list         # [n] arrays of positions
    upper: dict          # (position, level) -> list of positions
    ext_ids: np.ndarray | None = None


def read_optimized(path) -> Saved:
    """Hnsw::SaveOptimizedIndex as csrc/hnsw_format.cpp writes it: the header, one record per node (external id,
    label, data length, row, level-0 count and links), then per node u32 bytes and its upper-level block of
    maxM + 1 ints per level (count, links)."""
    import struct
    raw = open(path, "rb").read()
    hdr = "<IIQQQiIQQiQ"
    _, n, mem_per, off_l0, _, maxlevel, enterpoint, maxM, maxM0, _, _ = struct.unpack_from(hdr, raw, 0)
    off = struct.calcsize(hdr)
    rec = np.frombuffer(raw, np.uint8, n * mem_per, off).reshape(n, mem_per)
    ext = rec[:, 0:4].copy().view(np.int32)[:, 0]
    cnt0 = rec[:, off_l0:off_l0 + 4].copy().view(np.int32)[:, 0].astype(np.int64)
    lk = rec[:, off_l0 + 4:off_l0 + 4 + 4 * maxM0].copy().view(np.int32)
    links0 = [lk[i, :cnt0[i]].astype(np.int64) for i in range(n)]
    off += n * mem_per
    levels = np.zeros(n, np.int64)
    upper = {}
    for i in range(n):
        (nbytes,) = struct.unpack_from("<I", raw, off)
        off += 4
        blk = np.frombuffer(raw, np.int32, nbytes // 4, off)
        off += nbytes
        levels[i] = nbytes // (4 * (maxM + 1))
        for l in range(1, levels[i] + 1):
            b = blk[(l - 1) * (maxM + 1):l * (maxM + 1)]
            upper[(i, l)] = b[1:1 + b[0]].tolist()
    assert off == len(raw), "trailing bytes after the upper-level blocks"
    return Saved(maxlevel, enterpoint, maxM, maxM0, levels, cnt0, links0, upper, ext)


def read_regular(path) -> Saved:
    """Hnsw::SaveRegularIndexBin (what a uint8 l2sqr_sift index saves): u32 0, u32 total, i32 maxlevel,
    u32 enterpoint, u64 M, maxM, maxM0, then per node u32 level and per level 0..level u32 count + links."""
    import struct
    raw = open(path, "rb").read()
    _, n, maxlevel, enterpoint, _, maxM, maxM0 = struct.unpack_from("<IIiIQQQ", raw, 0)
    off = struct.calcsize("<IIiIQQQ")
    levels = np.zeros(n, np.int64)
    cnt0 = np.zeros(n, np.int64)
    links0, upper = [], {}
    for i in range(n):
        (levels[i],) = struct.unpack_from("<I", raw, off)
        off += 4
        for l in range(levels[i] + 1):
            (c,) = struct.unpack_from("<I", raw, off)
            lst = np.frombuffer(raw, np.int32, c, off + 4).astype(np.int64)
            off += 4 + 4 * c
            if l == 0:
                cnt0[i] = c
                links0.append(lst)
            else:
                upper[(i, l)] = lst.tolist()
    assert off == len(raw), "trailing bytes after the last node"
    return Saved(maxlevel, enterpoint, maxM, maxM0, levels, cnt0, links0, upper)


def case_params(case: Case) -> dict:
    p = {"M": 16, "efConstruction": 200}
    p.update(case.params)
    return p


_ROWS: dict = {}
_GRAPHS: dict = {}


def case_rows(case: Case):
    if case.name not in _ROWS:
        _ROWS[case.name] = case.rows()
    return _ROWS[case.name]


def restated(case: Case, levels) -> Graph:
    """The restated graph of a case for the given levels (kept for the session: the CPU and GPU tests share it)."""
    levels = np.asarray(levels, np.int64)
    key = (case.name, levels.tobytes())
    if key not in _GRAPHS:
        p = case_params(case)
        _GRAPHS[key] = restate(case.space, case_rows(case), levels, p["M"], p["efConstruction"], p.get("maxM"),
                               p.get("maxM0"))
    return _GRAPHS[key]
