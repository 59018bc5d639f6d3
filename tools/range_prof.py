"""Timing of the batched range queries (nmslib_b200_range_query_batch, K5b) against the per-query range path.

usage: range_prof.py [--n N] [--u8-n U] [--nq Q] [--sample S] [--shapes l2,cosinesimil,u8,l1,linf] [--out FILE]

Five shapes: n x 128 l2 (TS kernel), n x 768 cosinesimil (pair kernel), U x 128 bytes l2sqr_sift
(synth.sift_like_u8, the integer-pipe kernel), and n x 128 l1 and linf (the CUDA-core scan K2 in range mode), Q queries
each, radius at the 10th and at the 100th neighbour of every query, capacity 128.  For each it reports the batch wall time (host in / host out), the pass-1 kernel time (CUDA
events, stats.last_scan_ms) and its rate (2 Q N D) against the stream peak DESIGN.md uses (TF32 1 108 TFLOP/s, INT8
3 780 TOP/s), the threshold and verification kernel times (torch.profiler, a separate run), the fallback count, and
the per-query rangeQuery time over S queries.  The uint8 shape also builds a second index with option force_exact=1,
which takes the per-query exact scan for every range query, and times a batch of the same S queries on it (checked
equal to the first index's answers), and so do l1 and linf, whose pass-1 rate is reported next to the rate of K2's
kNN pass (k = 10) over the same index and queries (no peak share: the CUDA-core scan has no data-sheet rate).  Prints
the GPU name and power limit first.
Defaults: n = 1 000 000, U = 10 000 000, Q = 10 000, S = 200."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import nmslib_zig_b200 as nb  # noqa: E402
from nmslib_zig_b200 import synth  # noqa: E402

TF32_PEAK = 1108.0  # TFLOP/s, DESIGN.md (tools/tc_peak.cu stream peak)
INT8_PEAK = 3780.0  # TOP/s, DESIGN.md (the low end of tools/tc_peak.cu's INT8 stream peak)
KERNELS = ("tc_range_threshold_u8", "tc_range_threshold", "tc_scan_ts", "tc_scan_pair", "tc_scan_u8", "scan_exact",
           "range_verify", "range_dist", "range_collect")  # (a name that contains another comes first)


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # (reported, not guessed)
        out = f"unavailable ({e})"
    return {"gpu": name, "power_limit_and_max_sm_clock": out}


def kernel_times(fn):
    """device time per kernel name (ms) of one call of fn, from torch.profiler with CUDA activities"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        t = getattr(ev, "device_time_total", 0)
        for key in KERNELS:
            if key in ev.name:
                out[key] = out.get(key, 0.0) + t / 1e3
                break
    return out


def make_index(space, data, **options):
    """options: process-wide, read when the index is created (restored to 0 afterwards)"""
    u8 = space == "l2sqr_sift"
    for k, v in options.items():
        nb.set_option(k, v)
    try:
        idx = nb.Index(space, None, "seq_search", "DenseUInt8Vector" if u8 else "DenseVector", "Int" if u8 else "Float")
    finally:
        for k in options:
            nb.set_option(k, 0)
    (idx.addUInt8Batch if u8 else idx.addDenseBatch)(data)
    idx.buildIndex()
    return idx


def no_device(what):
    # (a CPU rehearsal gets this far: arguments, data, index construction)
    raise SystemExit(f"range_prof.py: {what} built; the measurements need a CUDA device, none is visible")


def run_shape(space, n, dim, nq, sample, emit):
    data = synth.uniform(n, dim, 3) - 0.3
    q = synth.uniform(nq, dim, 4) - 0.3
    idx = make_index(space, data)
    if not nb.device_available():
        no_device(f"{space} {n}x{dim} index")
    for rec, _, _ in measure(idx, space, q, n, dim, sample, TF32_PEAK):
        emit(rec)
    idx.deinit()


def run_u8(n, nq, sample, emit):
    data, q = synth.sift_like_u8(n, 3), synth.sift_like_u8(nq, 4)
    idx = make_index("l2sqr_sift", data)
    exact = make_index("l2sqr_sift", data, force_exact=1)
    if not nb.device_available():
        no_device(f"l2sqr_sift {n}x128 indexes (integer pipe, force_exact=1)")
    for rec, r, radii in measure(idx, "l2sqr_sift", q, n, 128, sample, INT8_PEAK):
        rec["u8_imma"] = idx.stats()["u8_imma"]
        emit(compare_force_exact(exact, q, r, radii, sample, rec))
    idx.deinit()
    exact.deinit()


def run_lp(space, n, nq, sample, emit):
    """l1 / linf: K2 in range mode; its pass-1 rate next to K2's kNN pass over the same index and queries"""
    data = synth.uniform(n, 128, 3) - 0.3
    q = synth.uniform(nq, 128, 4) - 0.3
    idx = make_index(space, data)
    exact = make_index(space, data, force_exact=1)
    if not nb.device_available():
        no_device(f"{space} {n}x128 indexes (K2 range mode, force_exact=1)")
    knn = []
    for _ in range(3):
        idx.knnQueryBatch(q, 10)
        knn.append(idx.stats()["last_scan_ms"])
    knn_ms = min(knn)
    flop = 2.0 * nq * n * 128
    for rec, r, radii in measure(idx, space, q, n, 128, sample, None):
        rec.update({"knn_k10_pass_ms": round(knn_ms, 4), "knn_k10_pass_tflops": round(flop / (knn_ms * 1e-3) / 1e12, 1)})
        emit(compare_force_exact(exact, q, r, radii, sample, rec))
    idx.deinit()
    exact.deinit()


def compare_force_exact(exact, q, r, radii, sample, rec):
    """time a batch of `sample` of the queries on an index created with force_exact=1 (the per-query exact scan for
    every query) and check its answers equal r's"""
    nq = len(q)
    pick = np.linspace(0, nq - 1, sample).astype(int)
    st0 = exact.stats()
    t0 = time.perf_counter()
    e = exact.rangeQueryBatch(q[pick], radii[pick], 128)
    wall = (time.perf_counter() - t0) * 1e3
    st = exact.stats()
    same = (np.array_equal(e.sizes, r.sizes[pick]) and np.array_equal(e.ids, r.ids[pick])
            and np.array_equal(e.distances.view(np.int32), r.distances[pick].view(np.int32)))
    rec.update({"force_exact_batch_queries": int(len(pick)), "force_exact_batch_ms": round(wall, 2),
                "force_exact_ms_per_query": round(wall / len(pick), 4),
                "force_exact_x_Q_ms": round(wall / len(pick) * nq, 1),
                "force_exact_tc_queries": int(st["range_tc_queries"] - st0["range_tc_queries"]),
                "force_exact_answers_equal": bool(same),
                "speedup_vs_force_exact": round(wall / len(pick) * nq / rec["batch_wall_ms"], 1)})
    return rec


def measure(idx, space, q, n, dim, sample, peak):
    """yields (record, the last batch's result, radii) per radius"""
    nq = len(q)
    kd = idx.knnQueryBatch(q, 100).distances
    for nth in (10, 100):
        radii = kd[:, nth - 1].astype(np.float64)
        idx.rangeQueryBatch(q, radii, 128)                      # warm-up (module load, scratch allocation)
        walls, scans = [], []
        for _ in range(3):
            st0 = idx.stats()
            t0 = time.perf_counter()
            r = idx.rangeQueryBatch(q, radii, 128)
            walls.append((time.perf_counter() - t0) * 1e3)
            st = idx.stats()
            scans.append(st["last_scan_ms"])
        fb = st["range_fallback_queries"] - st0["range_fallback_queries"]
        tcq = st["range_tc_queries"] - st0["range_tc_queries"]
        ktimes = kernel_times(lambda: idx.rangeQueryBatch(q, radii, 128))
        pick = np.linspace(0, nq - 1, sample).astype(int)
        idx.rangeQuery(q[pick[0]], float(radii[pick[0]]), capacity=128)
        t0 = time.perf_counter()
        for i in pick:
            idx.rangeQuery(q[i], float(radii[i]), capacity=128)
        per_q = (time.perf_counter() - t0) * 1e3 / len(pick)
        pass1 = min(scans)
        flop = 2.0 * nq * n * dim
        unit, pipe = ("tops", "int8") if peak == INT8_PEAK else ("tflops", "tf32")
        rec = {"space": space, "n": n, "dim": dim, "nq": nq, "radius_at_neighbour": nth, "capacity": 128,
               "batch_wall_ms": round(min(walls), 3), "pass1_ms": round(pass1, 4),
               f"pass1_{unit}": round(flop / (pass1 * 1e-3) / 1e12, 1) if pass1 > 0 else None}
        if peak:
            rec[f"pass1_share_of_{pipe}_peak"] = round(flop / (pass1 * 1e-3) / 1e12 / peak, 3) if pass1 > 0 else None
        rec.update({"kernel_ms_profiler": {k: round(v, 4) for k, v in ktimes.items()},
                    "tc_queries": int(tcq), "fallback_queries": int(fb),
                    "mean_hits": round(float(r.sizes.mean()), 2),
                    "single_query_ms": round(per_q, 4), "single_query_x_Q_ms": round(per_q * nq, 1),
                    "speedup_vs_single": round(per_q * nq / min(walls), 1)})
        yield rec, r, radii


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--u8-n", type=int, default=10_000_000)
    ap.add_argument("--nq", type=int, default=10_000)
    ap.add_argument("--sample", type=int, default=200)
    ap.add_argument("--shapes", default="l2,cosinesimil,u8")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = []

    def emit(rec):
        s = json.dumps(rec)
        print(s, flush=True)
        lines.append(s)

    if nb.device_available():
        emit(gpu_info())
    shapes = a.shapes.split(",")
    if "l2" in shapes:
        run_shape("l2", a.n, 128, a.nq, a.sample, emit)
    if "cosinesimil" in shapes:
        run_shape("cosinesimil", a.n, 768, a.nq, a.sample, emit)
    if "u8" in shapes:
        run_u8(a.u8_n, a.nq, a.sample, emit)
    for space in ("l1", "linf"):
        if space in shapes:
            run_lp(space, a.n, a.nq, a.sample, emit)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
