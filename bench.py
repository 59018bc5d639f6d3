#!/usr/bin/env python
"""bench.py -- queries/sec of the knnQueryBatch hot path on BASELINE.json's metric config.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic queries (config 2: 10 000
queries x 128-D against 1 000 000 x 128-D, l2sqr, k = 10).  Ours: `value` is measured with the
queries already resident in HBM (CUDA events on the launching stream, max over ranks);
`e2e` is the same batch through the C ABI with HOST buffers (H2D + kernels + D2H inside the
timed region).  N > 1 (torchrun, one rank per GPU): the database is row-sharded, every rank
scans its shard, the per-shard (key, id) lists are all-gathered over NCCL/NVLink and merged on
device (strong scaling of the fixed 1 M-row workload).
`--impl reference` times the reference's own CPU implementation (oracle/_ref: the unmodified
NMSLIB sources, OpenMP over queries on all host cores) on a bounded query sample of the same
workload.  Prints ONE JSON line on rank 0.
`--dump-outputs DIR` writes the answers of the last timed step of every record (the ids and distances a
caller of knnQueryBatch receives) to DIR, so that two builds can be compared output for output on the same
seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "queries/sec (k=10, exact & HNSW recall@10>=0.95) at 1/2/4/8 B200 vs CPU"
DUMP_LIMIT = 64 << 20       # bytes written by --dump-outputs, all records together
OUTPUTS = {}                # workload -> (ids, distances) of its last timed step, kept on rank 0 for --dump-outputs


def dump_outputs(out_dir: str, outputs: dict) -> None:
    """DIR/<workload>_ids.npy (float64, every int32 id exactly) and DIR/<workload>_distances.npy (float32), one row per
    query, and DIR/<workload>_rows.npy, the query rows they hold: all of them, or above DUMP_LIMIT in all the same
    fraction of every record's rows, chosen with a fixed seed."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    headers = 3 * 128 * len(outputs)                                  # .npy headers
    need = sum(ids.shape[0] * (12 * ids.shape[1] + 8) for ids, _ in outputs.values())
    frac = min(1.0, (DUMP_LIMIT - headers) / max(1, need))
    for name, (ids, dists) in outputs.items():
        nq = ids.shape[0]
        rows = np.arange(nq)
        if frac < 1.0:
            rows = np.sort(np.random.default_rng(0).choice(nq, int(nq * frac), replace=False))
            ids, dists = ids[rows], dists[rows]
        np.save(out / f"{name}_rows.npy", rows.astype(np.float64))
        np.save(out / f"{name}_ids.npy", ids.astype(np.float64))
        np.save(out / f"{name}_distances.npy", dists.astype(np.float32))


def keep_outputs(name: str, ids, dists, rank: int, world: int, sliced: bool) -> None:
    """Copy a record's device answers to the host after its timed steps, for --dump-outputs.  sliced: every rank holds
    the answers of its own slice of the batch (hnsw replicas) and rank 0 joins them; otherwise rank 0 holds them all."""
    if sliced and world > 1:
        import torch.distributed as dist
        parts = [None] * world if rank == 0 else None
        dist.gather_object((ids.cpu().numpy(), dists.cpu().numpy()), parts, dst=0)
        if rank == 0:
            OUTPUTS[name] = (np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]))
    elif rank == 0:
        OUTPUTS[name] = (ids.cpu().numpy(), dists.cpu().numpy())


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.device)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def workload(name: str, n: int | None, nq: int | None, rank: int = 0, world: int = 1):
    """The config's synthetic data; with world > 1 only this rank's row shard of it (w["lo"], w["hi"])."""
    from nmslib_zig_b200 import synth
    from nmslib_zig_b200.shard import shard_bounds
    space, method, dtype, dist, n0, dim, nq0, k, _, _ = synth.CONFIGS[name]
    n = n or n0
    lo, hi = shard_bounds(n, rank, world)
    data, queries = synth.make(name, n, nq, rows=(lo, hi) if world > 1 else None)
    return dict(name=name, space=space, method=method, dtype=dtype, dist=dist, dim=dim, k=k, data=data,
                queries=queries, n=n, nq=queries.shape[0], lo=lo, hi=hi, full_size=(n == n0 and queries.shape[0] == nq0))



def sample_queries(nq: int, want: int) -> np.ndarray:
    """Indices of `want` queries spread evenly over the batch (every 256-query block of the scan is represented
    as far as `want` allows)."""
    return np.unique(np.linspace(0, nq - 1, min(want, nq)).astype(np.int64))


def parity_seq(w, sel, got_ids, got_dists, rank, world, dist_on, threads=None):
    """Check the final (merged) answers of the queries `sel` against the oracle (oracle/knn_oracle.c, the CPU
    restatement of SeqSearch::Search + the distance kernels, pinned to the reference by tests/test_oracle.py).
    N > 1: every rank runs the oracle over ITS OWN row shard (w["data"] holds nothing else), the per-shard oracle
    lists go to rank 0 over the host channel and are merged there by (distance, global position) -- the
    specification of the device merge (nmslib_zig_b200/shard.py).  Returns the `parity` record on rank 0."""
    from oracle import oracle as O
    sys.path.insert(0, str(ROOT / "tests"))
    from helpers import ATOL_COSINE, RTOL, ATOL, count_mismatches
    from nmslib_zig_b200.shard import make_keys
    k, space = w["k"], w["space"]
    u8 = w["dtype"] == "DenseUInt8Vector"
    t0 = time.perf_counter()
    pos = np.arange(w["lo"], w["hi"], dtype=np.int32)
    thr = threads or max(1, (os.cpu_count() or 1) // world)
    oi, od, oc = O.seq_knn(space, w["data"], w["queries"][sel], k, pos, threads=thr)
    if dist_on:
        import torch.distributed as dist
        gathered = [None] * world if rank == 0 else None
        dist.gather_object((oi, od), gathered, dst=0)
        if rank != 0:
            return None
        allp = np.concatenate([g[0] for g in gathered], axis=1)               # [q, world * k] global positions
        alld = np.concatenate([g[1] for g in gathered], axis=1)
        order = np.argsort(make_keys(alld, allp), axis=1, kind="stable")[:, :k]   # (distance, position) order
        oi = np.take_along_axis(allp, order, axis=1)
        od = np.take_along_axis(alld, order, axis=1)
        oc = (oi >= 0).sum(axis=1).astype(np.int32)
    gi, gd = np.asarray(got_ids)[sel], np.asarray(got_dists)[sel]
    gc = (gi >= 0).sum(axis=1).astype(np.int32)
    bad = count_mismatches(gi, gd, gc, oi, od, oc, exact=u8, atol=ATOL_COSINE if space == "cosinesimil" else None)
    return {"checked": int(len(sel)), "mismatches": int(bad), "against": "oracle/knn_oracle.c over all "
            f"{w['n']} rows" + (f" ({world} shard oracles merged on the host)" if dist_on else ""),
            "tolerance": "bit-exact ids and distances (ties: set-equal)" if u8 else
                         f"ids exact outside tie groups; |d - d_ref| <= {RTOL}*|d_ref| + {ATOL}",
            "seconds": time.perf_counter() - t0}


def synth_method(name: str) -> str:
    from nmslib_zig_b200 import synth
    return synth.CONFIGS[name][1]


def ref_space(space):  # l2sqr is not a registered reference space (SURVEY 0.3): same ranking as l2
    return "l2" if space == "l2sqr" else space


def time_reference(w, sample: int, steps: int, warmup: int):
    """The reference's CPU path on `sample` queries per step, OpenMP over queries on all cores."""
    from oracle import oracle as O
    threads = os.cpu_count() or 1
    q = w["queries"][:sample]
    if O.ref_available():
        kind = "reference"
        ref = O.RefIndex(ref_space(w["space"]), "seq_search").add(w["data"]).build("")
        run = lambda: ref.knn(q, w["k"], threads=threads)
    else:
        kind = "port"
        run = lambda: O.seq_knn(w["space"], w["data"], q, w["k"], threads=threads)
    for _ in range(warmup):
        run()
    t0 = time.perf_counter()
    for _ in range(steps):
        run()
    dt = (time.perf_counter() - t0) / steps
    # SURVEY 8d (A): the path as shipped -- lib.zig calls nmslib_knn_query_fill in a serial loop, one core
    one = None
    if kind == "reference":
        q1 = q[:min(32, sample)]
        t1 = time.perf_counter()
        ref.knn(q1, w["k"], threads=1)
        one = len(q1) / (time.perf_counter() - t1)
    return {"value": sample / dt, "unit": "queries/s", "cores": threads, "kind": kind, "as_shipped_1core": one,
            "sample": f"{sample} of {w['nq']} queries x all {w['n']} rows per step, {steps} steps"
                      + (" (space l2: l2sqr is not registered in the reference; same ranking + one sqrtf)"
                         if w["space"] == "l2sqr" else ""),
            "ms_per_step": dt * 1e3}


def run_hnsw(args, w, rank, world, local_rank, dev, dist_on, n_steps, with_cpu):
    """Config 3: HNSW beam search (K3).  One graph does not shard without changing its answers (SURVEY 8e): every
    rank holds a replica of the index -- built on the device by csrc/hnsw_build_gpu.cu -- and takes 1/N of the
    queries; there is no data-path collective.  efSearch = the smallest of the sweep that reaches recall@10 >= 0.95
    against the exact scan on a query sample (the metric's condition), else the largest."""
    import torch
    import nmslib_zig_b200 as nb
    if dist_on:
        import torch.distributed as dist
    n, nq, dim, k = w["n"], w["nq"], w["dim"], w["k"]
    data, queries = w["data"], w["queries"]
    t0 = time.perf_counter()
    idx = nb.Index(w["space"], None, "hnsw")
    idx.addDenseBatch(data)
    idx.buildIndex(nb.Params({"M": 16, "efConstruction": 200, "b200_build": "device"}))
    idx.prepare()
    build_s = time.perf_counter() - t0
    build = {k_: v for k_, v in idx.stats().items() if k_.startswith("build_")}
    # ground truth for the recall condition: the exact scan (itself parity-tested) on a query sample
    sample = queries[:: max(1, nq // 1000)][:1000]
    ex = nb.Index(w["space"], None, "seq_search")
    ex.addDenseBatch(data)
    ex.buildIndex()
    exact_ids = ex.knnQueryBatch(sample, k).ids
    ex.deinit()
    sweep, ef, rec = [], None, 0.0
    for cand in (50, 100, 200, 400, 800):
        idx.setQueryTimeParams(nb.Params({"efSearch": cand}))
        got = idx.knnQueryBatch(sample, k).ids
        r = float(np.mean([len(set(a.tolist()) & set(b.tolist())) / k for a, b in zip(got, exact_ids)]))
        sweep.append({"efSearch": cand, "recall": r})
        ef, rec = cand, r
        if r >= 0.95:
            break
    idx.setQueryTimeParams(nb.Params({"efSearch": ef}))
    q_lo, q_hi = (nq * rank) // world, (nq * (rank + 1)) // world
    my_nq = q_hi - q_lo
    q_host = torch.from_numpy(np.ascontiguousarray(queries[q_lo:q_hi])).pin_memory()
    d_q = q_host.to(dev)
    d_ids = torch.empty((my_nq, k), dtype=torch.int32, device=dev)
    d_dists = torch.empty((my_nq, k), dtype=torch.float32, device=dev)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)

    def step_device():
        idx.knnDevice(d_q.data_ptr(), my_nq, dim, k, d_ids.data_ptr(), d_dists.data_ptr(), 0, stream.cuda_stream)

    def barrier():
        if dist_on:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        step_device()
    barrier()
    st0 = idx.stats()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(n_steps):
        step_device()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    st1 = idx.stats()
    if args.dump_outputs:
        keep_outputs(w["name"], d_ids, d_dists, rank, world, sliced=True)
    q_np = q_host.numpy()
    for _ in range(2):
        idx.knnQueryBatch(q_np, k)
    barrier()
    t0 = time.perf_counter()
    for _ in range(n_steps):
        idx.knnQueryBatch(q_np, k)
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / n_steps
    if dist_on:
        t = torch.tensor([ms, e2e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = float(t[0].item()), float(t[1].item())
    clocks = sampler.stop() if rank == 0 else None
    line = None
    if rank == 0:
        peaks = load_peaks()
        ms_per_step = ms / n_steps
        steps = max(1, n_steps)
        evals = (st1["distance_evals"] - st0["distance_evals"]) / steps
        exps = (st1["hnsw_expansions"] - st0["hnsw_expansions"]) / steps
        kern_ms = (st1["scan_ms_sum"] - st0["scan_ms_sum"]) / max(1, st1["scan_count"] - st0["scan_count"])
        launches_per_step = (st1["scan_count"] - st0["scan_count"]) / steps
        gbytes = (evals * 4.0 * dim + exps * 4.0 * 32) / 1e9          # SURVEY 8d: rows gathered + adjacency lists read
        achieved = gbytes / max(1e-9, kern_ms * launches_per_step * 1e-3)
        traffic = None
        try:  # DRAM bytes per launch from the committed ncu capture (full-size config, one GPU, efSearch 400 only)
            tj = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "traffic.json")))
            if world == 1 and w["full_size"] and ef == 400 and w["name"] in tj:
                traffic = tj[w["name"]]["bytes"]
        except Exception:
            traffic = None
        cpu, parity = None, None
        if world == 1 and with_cpu:
            # the REFERENCE's own HNSW search (Index::LoadIndex + Search through oracle/_ref, OpenMP over queries on all
            # host cores) on the SAME device-built graph, same efSearch, a bounded query sample
            from oracle import oracle as O
            if O.ref_available():
                threads = os.cpu_count() or 1
                ref = O.RefIndex(w["space"], "hnsw")
                with tempfile.TemporaryDirectory() as tmp:
                    path = os.path.join(tmp, "c3.hnsw")
                    idx.save(path, False)
                    ref.load(path)
                ref.set_query_params(f"efSearch={ef}")
                ref.knn(sample[:64], k, threads=threads)
                t0 = time.perf_counter()
                ri, _, _ = ref.knn(sample, k, threads=threads)
                dt = time.perf_counter() - t0
                rec_ref = float(np.mean([len(set(a.tolist()) & set(b.tolist())) / k for a, b in zip(ri, exact_ids)]))
                # north_star: recall@10 at or above the reference HNSW's at the same efSearch on the same graph; the ids
                # themselves agree except where fp32 rounding reorders near-ties inside the beam
                agree = float(np.mean([len(set(a.tolist()) & set(b.tolist())) / k for a, b in zip(got, ri)]))
                parity = {"checked": int(len(sample)), "mismatches": int(rec < rec_ref - 2e-3),
                          "recall_ours": rec, "recall_reference_same_graph": rec_ref, "id_agreement_with_reference": agree,
                          "against": "the reference's Hnsw::Search (oracle/_ref) on the same graph at the same efSearch; "
                                     "ground truth for recall = this library's exact scan (itself checked against the oracle)",
                          "tolerance": "recall_ours >= recall_reference - 2e-3"}
                cpu = {"value": len(sample) / dt, "unit": "queries/s", "cores": threads, "kind": "reference",
                       "sample": f"{len(sample)} of {nq} queries, the reference's Hnsw::Search on the same (device-built) "
                                 f"graph at efSearch={ef}; its recall@{k} on that sample: {rec_ref:.4f} (ours: {rec:.4f})"}
                ref.close()
        line = {
            "metric": METRIC, "value": nq / (ms_per_step * 1e-3), "unit": "queries/s", "n_gpus": world,
            "steps": n_steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{w['name']}: hnsw {w['space']} {n}x{dim}, M=16 efConstruction=200 (graph built on the "
                                   f"device), efSearch={ef}, {nq} queries, k={k}", "space": w["space"], "k": k,
                       "efSearch": ef, "recall_at_k": rec, "recall_sweep": sweep,
                       "parallelism": f"index replicated x{world}, queries split {world} ways (no collective)",
                       "l2_policy": f"random gathers over {n * dim * 4 / 1e6:.0f} MB of rows (L2 is 126 MB)",
                       "build_s_incl_upload": build_s, **build},
            "e2e": {"value": nq / (e2e_ms * 1e-3), "unit": "queries/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(nq * dim * 4), "d2h_bytes_per_step": int(nq * k * 8 + nq * 4)},
            "gpu_launches": int(st1["kernel_launches"] - st0["kernel_launches"]),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": achieved / peaks["hbm_gbs"], "traffic": traffic, "kernel": "hnsw_search",
                         "kernel_ms": kern_ms * launches_per_step,
                         "bytes_per_query": gbytes * 1e9 / max(1, my_nq),
                         "peak_src": f"{peaks['src']} HBM copy bandwidth"},
            "parity": parity, "cpu_baseline": cpu, "clocks": clocks,
        }
    idx.deinit()
    return line if rank == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--n", "--rows", dest="n", type=int, default=None,
                    help="override database rows (debug; under torchrun use --rows: its parser claims --n)")
    ap.add_argument("--nq", type=int, default=None, help="override query count (debug)")
    ap.add_argument("--cpu-sample", type=int, default=1024)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--workloads", default="c1,c4,c3",
                    help="further single-GPU configs reported as sub-records of the default line ('none' to skip)")
    ap.add_argument("--budget-s", type=float, default=420.0, help="no new sub-record is started after this many seconds")
    ap.add_argument("--parity-sample", type=int, default=256, help="queries of the final answer checked against the oracle")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: 'peer' = the library's own NVLink peer-memory exchange, 'nccl' = all-gather + merge")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the ids and distances of every record's last timed step to DIR as .npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the answers of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        w = workload(args.workload, args.n, args.nq)
        sample = min(args.cpu_sample // 2, w["nq"])
        base = time_reference(w, sample, max(1, args.steps), max(0, args.warmup))
        line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": "queries/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": base["ms_per_step"],
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": f"{w['name']}: seq_search {w['space']} {w['n']}x{w['dim']}, "
                                       f"{w['nq']} queries, k={w['k']}", "space": w["space"], "k": w["k"]},
                "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample", "as_shipped_1core")},
                "e2e": {"value": base["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ our arm (GPU)
    import torch
    import nmslib_zig_b200 as nb

    if not torch.cuda.is_available() or not nb.device_available():
        raise SystemExit("bench.py: no CUDA device -- the query path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    nb.set_device(local_rank)
    dist_on = world > 1
    if dist_on:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    t_start = time.perf_counter()

    def run(name, n=None, nq=None, steps=None, warmup=None, cpu=True):
        if synth_method(name) == "hnsw":          # config 3: replicas, queries split (no row shards)
            w = workload(name, n, nq)
            return run_hnsw(args, w, rank, world, local_rank, dev, dist_on, steps or args.steps, cpu and not args.no_cpu)
        w = workload(name, n, nq, rank, world)
        return run_seq(args, w, rank, world, local_rank, dev, dist_on, steps or args.steps, warmup or args.warmup,
                       cpu and not args.no_cpu)

    line = run(args.workload, args.n, args.nq)
    # the other single-GPU configurations of BASELINE.json as sub-records of the default line (driver-visible parity,
    # roofline and cpu_baseline for each): config 1, config 4 at full size, config 3 at full size
    subs = [x for x in args.workloads.split(",") if x and x != "none" and x != args.workload]
    if world == 1 and args.n is None and args.nq is None and subs and line is not None:
        line["workloads"] = {}
        for name in subs:
            if time.perf_counter() - t_start > args.budget_s:
                line["workloads"][name] = {"skipped": f"time budget of {args.budget_s:.0f} s spent"}
                continue
            try:
                rec = run(name, warmup=3)
                for drop in ("metric", "unit", "higher_is_better", "vs_baseline", "data", "n_gpus", "clocks"):
                    rec.pop(drop, None)
                line["workloads"][name] = rec
            except Exception as e:  # a sub-record must not take the headline line down with it
                line["workloads"][name] = {"error": f"{type(e).__name__}: {e}"}
    # several GPUs, default run: config 4 (10 M x 128 uint8, the integer tensor pipe) sharded the same way as a
    # sub-record -- the bit-exact parity sample over all 10 M rows at every N (every rank makes the same calls)
    if (world > 1 and args.workload == "c2" and args.n is None and args.nq is None and "c4" in subs
            and time.perf_counter() - t_start < args.budget_s):
        rec = None
        try:
            rec = run("c4", warmup=3, cpu=False)
        except Exception as e:
            rec = {"error": f"{type(e).__name__}: {e}"}
        if rank == 0 and line is not None and rec is not None:
            for drop in ("metric", "unit", "higher_is_better", "vs_baseline", "data", "n_gpus", "clocks"):
                rec.pop(drop, None)
            line.setdefault("workloads", {})["c4"] = rec
    # config 5 (10 M x 768 negdotprod, 100 K queries, k = 100) is the one BASELINE configuration that needs the whole
    # box: on the default 8-GPU run it is reported as a sub-record, with its own parity sample, next to config 2
    if (world == 8 and args.workload == "c2" and args.n is None and args.nq is None and "none" not in args.workloads
            and time.perf_counter() - t_start < args.budget_s):
        rec = None
        try:
            args.parity_sample = min(args.parity_sample, 64)
            rec = run("c5", warmup=3, cpu=False)
        except Exception as e:
            rec = {"error": f"{type(e).__name__}: {e}"}
        if rank == 0 and line is not None and rec is not None:
            for drop in ("metric", "unit", "higher_is_better", "vs_baseline", "data", "n_gpus", "clocks"):
                rec.pop(drop, None)
            line.setdefault("workloads", {})["c5"] = rec
    if rank == 0 and line is not None:
        line["wall_s"] = time.perf_counter() - t_start
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, OUTPUTS)
        print(json.dumps(line))
    if dist_on:
        dist.destroy_process_group()


def run_seq(args, w, rank, world, local_rank, dev, dist_on, steps, warmup, with_cpu):
    """Sequential-search workloads (configs 1, 2, 4, 5): one rank per GPU, rows sharded, the per-shard key lists
    exchanged and merged on the device every step.  Returns the JSON record on rank 0 (None elsewhere)."""
    import torch
    import nmslib_zig_b200 as nb
    if dist_on:
        import torch.distributed as dist
    n, nq, dim, k = w["n"], w["nq"], w["dim"], w["k"]
    u8 = w["dtype"] == "DenseUInt8Vector"
    lo, hi = w["lo"], w["hi"]
    # (the CUDA context, the library's stream and its upload kernels exist before the ingest clock starts: a throw-away
    # index of the same kind goes through the same calls once)
    torch.zeros(1, device=dev)
    tiny = nb.Index(w["space"], None, w["method"], w["dtype"], w["dist"])
    (tiny.addUInt8Batch if u8 else tiny.addDenseBatch)(w["data"][:256])
    tiny.buildIndex()
    tiny.prepare()
    tiny.deinit()
    idx = nb.Index(w["space"], None, w["method"], w["dtype"], w["dist"])
    idx.setShard(lo)                                   # keys carry GLOBAL positions (tie order, SURVEY 8e)
    shard_ids = np.arange(lo, hi, dtype=np.int32)
    t_ing = time.perf_counter()
    (idx.addUInt8Batch if u8 else idx.addDenseBatch)(w["data"], shard_ids)   # (w["data"] is this rank's shard)
    t_add = time.perf_counter() - t_ing
    idx.buildIndex()
    idx.prepare()                                      # upload + operand preparation (SURVEY 8f N2: the ingest path)
    t_ing = time.perf_counter() - t_ing
    ingest = {"rows": int(hi - lo), "seconds": t_ing, "add_seconds": t_add, "rows_per_s": (hi - lo) / t_ing,
              "gbytes_per_s": w["data"].nbytes / t_ing / 1e9,
              "what": "nmslib_add_data_point_batch (one slab copy on the host) + upload + operand preparation, one rank; CUDA context and kernels loaded beforehand by a 256-row index"}

    q_host = torch.from_numpy(w["queries"]).pin_memory()
    d_q = q_host.to(dev, non_blocking=False)
    d_ids = torch.empty((nq, k), dtype=torch.int32, device=dev)
    d_dists = torch.empty((nq, k), dtype=torch.float32, device=dev)
    d_keys = torch.empty((nq, k), dtype=torch.int64, device=dev)
    exchange = "none"
    if dist_on:
        exchange = args.exchange
        if exchange == "peer":
            # the library's own exchange: every rank exports its key window (CUDA IPC), the 128-byte blobs travel over
            # the host channel once, then nmslib_b200_knn_device returns the GLOBAL top-k on every rank with no
            # collective call per step (publish + merge over NVLink peer memory inside the engine's stream)
            try:
                blob = idx.shardExport(nq, k)
                blobs = [None] * world
                dist.all_gather_object(blobs, bytes(blob))
                idx.shardConnect(rank, world, b"".join(blobs))
            except Exception as e:
                if rank == 0:
                    print(f"bench.py: peer exchange unavailable ({e}); falling back to NCCL all-gather", file=sys.stderr)
                exchange = "nccl"
            flag = torch.tensor([1 if exchange == "peer" else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)     # all ranks or none
            if int(flag.item()) == 0 and exchange == "peer":
                idx.shardDisconnect()
                exchange = "nccl"
        if exchange == "nccl":
            g_keys = torch.empty((world, nq, k), dtype=torch.int64, device=dev)
            o_ids = torch.empty((nq, k), dtype=torch.int32, device=dev)
            o_dists = torch.empty((nq, k), dtype=torch.float32, device=dev)
        else:
            o_ids, o_dists = d_ids, d_dists
    # a dedicated non-default stream: the C ABI treats a NULL stream as "the engine's own stream", and CUDA
    # events only see the stream they are recorded on
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)

    def step_device():
        idx.knnDevice(d_q.data_ptr(), nq, dim, k, d_ids.data_ptr(), d_dists.data_ptr(), d_keys.data_ptr(),
                      stream.cuda_stream)
        if dist_on and exchange == "nccl":
            # the shards number their rows by global position (shard_ids above), which is what the keys carry: only
            # the (distance, position) keys cross NVLink, 8 bytes per candidate, and the merge takes the ids from them
            dist.all_gather_into_tensor(g_keys, d_keys)
            idx.mergeTopk(g_keys.data_ptr(), 0, world, nq, k, o_ids.data_ptr(), o_dists.data_ptr(), stream.cuda_stream)

    def barrier():
        if dist_on:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(warmup):
        step_device()
    barrier()
    st0 = idx.stats()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(steps):
        step_device()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs:
        keep_outputs(w["name"], o_ids if dist_on else d_ids, o_dists if dist_on else d_dists, rank, world, sliced=False)
    if dist_on:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    st1 = idx.stats()
    ms_per_step = ms / steps
    value = nq / (ms_per_step * 1e-3)
    launches = int(st1["kernel_launches"] - st0["kernel_launches"]) + (steps if exchange == "nccl" else 0)  # (+ the merge)
    scan_ms = (st1["scan_ms_sum"] - st0["scan_ms_sum"]) / max(1, st1["scan_count"] - st0["scan_count"])

    # ---- end to end through the public API: pinned host queries in, host results out ----
    q_np = q_host.numpy()
    if not dist_on:
        def step_e2e():
            return idx.knnQueryBatch(q_np, k)
        d2h = nq * k * 8 + nq * 4
    else:
        h_ids = torch.empty((nq, k), dtype=torch.int32).pin_memory()
        h_dists = torch.empty((nq, k), dtype=torch.float32).pin_memory()

        def step_e2e():
            d_q.copy_(q_host, non_blocking=True)
            step_device()
            if rank == 0:
                h_ids.copy_(o_ids, non_blocking=True)
                h_dists.copy_(o_dists, non_blocking=True)
            torch.cuda.synchronize(dev)
        d2h = nq * k * 8
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        res = step_e2e()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / steps
    if dist_on:
        t = torch.tensor([e2e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    st2 = idx.stats()

    # ---- parity of the final answers (every N): a query sample spread over all query blocks against the oracle ----
    if dist_on:
        got_ids, got_d = (h_ids.numpy(), h_dists.numpy()) if rank == 0 else (None, None)
    else:
        got_ids, got_d = res.ids, res.distances
    parity = parity_seq(w, sample_queries(nq, args.parity_sample), got_ids, got_d, rank, world, dist_on)

    line = None
    if rank == 0:
        peaks = load_peaks()
        ops = 2.0 * nq * (hi - lo) * dim                       # SURVEY 8d: 2*Q*N*D per launch (this rank's shard)
        achieved = ops / (scan_ms * 1e-3) / 1e12 if scan_ms > 0 else 0.0
        imma = bool(u8 and st2.get("u8_imma", 0))
        sustained = ms > 1000.0                                # a long timed region sits under the power cap
        peak, peak_src = tensor_peak(peaks, "i8" if imma else "tf32", sustained)
        cpu = None
        if with_cpu and world == 1:
            cpu = cpu_baseline_seq(w, args.cpu_sample)
        traffic = None
        try:  # DRAM bytes per launch from the committed ncu capture of this workload (full-size, one GPU only)
            tj = json.load(open(ROOT / "profiles" / "traffic.json"))
            if world == 1 and w["full_size"] and w["name"] in tj:
                traffic = tj[w["name"]]["bytes"]
        except Exception:
            traffic = None
        line = {
            "metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": world, "steps": steps,
            "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None,
            "dtype": ("u8 (integer tensor pipe, exact int32 distances)" if imma else
                      "u8 (widened to tf32 operands, exact integer sums in f32)") if u8 else "f32",
            "data": "synthetic",
            "config": {"workload": f"{w['name']}: {w['method']} {w['space']} {n}x{dim}, {nq} queries, k={k}",
                       "space": w["space"], "k": k, "rows_per_gpu": hi - lo,
                       "parallelism": f"row-sharded x{world}" + (
                           " + key exchange over NVLink peer memory + device k-way merge inside the library"
                           if exchange == "peer" else " + NCCL all-gather + device k-way merge" if dist_on else ""),
                       "l2_policy": f"inputs larger than L2 ({(hi - lo) * dim * (1 if u8 else 4) / 1e6:.0f} MB scanned per step)"},
            "e2e": {"value": nq / (e2e_ms * 1e-3), "unit": "queries/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(q_np.nbytes), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": launches, "ingest": ingest,
            "uncertified_queries_per_step": (st1["fallback_queries"] - st0["fallback_queries"]) / steps,
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TOP/s" if imma else "TFLOP/s",
                         "frac": achieved / peak, "traffic": traffic, "kernel": "scan", "kernel_ms": scan_ms,
                         "peak_src": peak_src},
            "parity": parity, "cpu_baseline": cpu, "clocks": clocks,
        }
    idx.deinit()
    return line


def tensor_peak(peaks, kind: str, sustained: bool):
    """Roofline denominator of the scan: the tcgen05 micro-benchmark of tools/tc_peak.cu run on this pool's B200s
    (profiles/r02_tc_peak.json: TF32 and INT8 MMA streams, operands resident, burst and sustained), as SURVEY 8d
    asks; falls back to the driver's bf16 measurement / 2 (TF32) or x 2 (INT8) when that file is missing."""
    try:
        tp = json.load(open(ROOT / "profiles" / "r02_tc_peak.json"))
        key = "tf32_m128n256k8_ts_cta1" if kind == "tf32" else "i8_m128n256k32_ts_cta1"
        v = tp[key]["sustained" if sustained else "burst"]
        return float(v), (f"tools/tc_peak.cu on this pool's B200 (profiles/r02_tc_peak.json): {kind} tcgen05 MMA stream, "
                          f"{'sustained' if sustained else 'burst'} {v:.0f} T(FL)OP/s")
    except Exception:
        base = peaks["bf16_tflops_sustained"] if sustained else peaks["bf16_tflops"]
        v = base / 2.0 if kind == "tf32" else base * 2.0
        return v, f"{peaks['src']} bf16 {'sustained' if sustained else 'burst'} {base} TF/s {'/ 2' if kind == 'tf32' else 'x 2'}"


def cpu_baseline_seq(w, cpu_sample: int):
    """The reference's CPU path on a bounded sample of the workload (about 10-30 s of CPU work).  Configs whose full
    scan would take minutes (10 M rows) are timed on a row subsample and scaled linearly in N -- seq_search costs
    exactly Q x N distance calls (SURVEY 8d)."""
    rows = w["n"]
    sub = w
    scale = 1.0
    if w["n"] > 2_000_000 and w["lo"] == 0 and w["hi"] == w["n"]:
        rows = 1_000_000
        sub = dict(w, data=w["data"][:rows], n=rows)
        scale = rows / w["n"]
    base = time_reference(sub, min(cpu_sample, w["nq"]), 3 if scale == 1.0 else 2, 1)
    out = {k_: base[k_] for k_ in ("value", "unit", "cores", "kind", "sample", "as_shipped_1core")}
    if scale != 1.0:
        out["value"] = base["value"] * scale
        if out["as_shipped_1core"]:
            out["as_shipped_1core"] *= scale
        out["sample"] += f"; timed on the first {rows} rows and scaled by {scale:g} to {w['n']} rows (cost is linear in N)"
    return out


if __name__ == "__main__":
    main()
