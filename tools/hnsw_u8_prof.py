"""K3 on uint8 rows (l2sqr_sift + hnsw): byte rows against another build of the library on the same graph.

    hnsw_u8_prof.py [--n 1000000] [--nq 10000] [--efs 50,100,200,400] [--reps 3] [--rounds 2]
                    [--other-lib PATH] [--evg-lib PATH] [--out profiles/r06_hnsw_u8_prof.jsonl]

Inputs: n x 128 sift_like_u8 rows (seed 7) and nq queries (seed 8).  The graph is built once on the device (M=16,
efConstruction=200) and saved as the reference's regular index file plus its .dat.  Each measurement runs in a child
process of its own (one library per process):
  - this tree's library loads the file (nmslib_load_index, uint8) and searches its byte rows;
  - --other-lib (e.g. a build of an earlier commit) adds the same rows and imports the same regular file;
  - --evg-lib (the -DNB200_EXPERIMENTS build) repeats this tree's search with NB200_HNSW_G = 2, 4 and 8 neighbours in
    flight per warp.
The two libraries alternate --rounds times.  Per efSearch: host-to-host queries/s (best of --reps batches),
last_scan_ms, recall@10 against the exact GPU seq_search, distance_evals and hnsw_expansions per query, bytes per query
(evals x row bytes + expansions x 4 x maxM0; row bytes 128, and 512 for the widened rows of --other-lib's uint8 path)
and GB/s over the kernel time.  The answers of every library must be identical, ids and distance bits, for every
query at every efSearch.  The card's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
MAXM0 = 32  # M = 16


def child_build(a):
    sys.path.insert(0, str(ROOT))
    import nmslib_zig_b200 as nb
    from nmslib_zig_b200 import synth
    data, q = synth.sift_like_u8(a.n, 7), synth.sift_like_u8(a.nq, 8)
    idx = nb.Index("l2sqr_sift", None, "hnsw", "DenseUInt8Vector", "Int")
    idx.addUInt8Batch(data)
    t0 = time.perf_counter()
    idx.buildIndex(nb.Params({"M": 16, "efConstruction": 200, "b200_build": "device"}))
    idx.save(a.graph)
    build_s = time.perf_counter() - t0
    idx.deinit()
    ex = nb.Index("l2sqr_sift", None, "seq_search", "DenseUInt8Vector", "Int")
    ex.addUInt8Batch(data)
    ex.buildIndex()
    r = ex.knnQueryBatch(q, 10)
    np.save(a.graph + ".exact.npy", r.ids)
    ex.deinit()
    print(json.dumps({"build_and_save_s": build_s}))


def child_search(a):
    sys.path.insert(0, str(ROOT))
    import nmslib_zig_b200 as nb
    from nmslib_zig_b200 import synth
    q = synth.sift_like_u8(a.nq, 8)
    try:
        import torch
        q = torch.from_numpy(q).pin_memory().numpy()
    except Exception:
        pass
    if a.mode == "import":                             # a library that imports the regular file over its own rows
        idx = nb.Index("l2sqr_sift", None, "hnsw", "DenseUInt8Vector", "Int")
        idx.addUInt8Batch(synth.sift_like_u8(a.n, 7))
        idx.importHnsw(a.graph)
    else:
        idx = nb.Index.load(a.graph, "DenseUInt8Vector", "Int")
    out, recs = {}, []
    for ef in [int(e) for e in a.efs.split(",")]:
        idx.setQueryTimeParams(nb.Params({"efSearch": ef}))
        idx.knnQueryBatch(q, 10)                       # warm-up of this shape
        best, scan = None, None
        for _ in range(a.reps):
            s0 = idx.stats()
            t0 = time.perf_counter()
            r = idx.knnQueryBatch(q, 10)
            dt = time.perf_counter() - t0
            s1 = idx.stats()
            if best is None or dt < best:
                best, scan = dt, s1["last_scan_ms"]
                evals = s1["distance_evals"] - s0["distance_evals"]
                exps = s1["hnsw_expansions"] - s0["hnsw_expansions"]
        out[f"ids{ef}"], out[f"d{ef}"] = r.ids, r.distances
        recs.append({"ef": ef, "host_qps": a.nq / best, "host_ms": best * 1e3, "last_scan_ms": scan,
                     "evals_per_q": evals / a.nq, "expansions_per_q": exps / a.nq,
                     "device_bytes": idx.stats()["device_bytes"]})
    np.savez(a.dump, **out)
    idx.deinit()
    print(json.dumps(recs))


def run_child(args, env_extra, what):
    env = dict(os.environ)
    env.update(env_extra)
    p = subprocess.run([sys.executable, __file__, *args], env=env, capture_output=True, text=True)
    if p.returncode != 0:
        sys.stderr.write(p.stdout + p.stderr)
        raise RuntimeError(f"{what} failed")
    return json.loads(p.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--nq", type=int, default=10_000)
    ap.add_argument("--efs", default="50,100,200,400")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--other-lib", default="")
    ap.add_argument("--evg-lib", default="")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r06_hnsw_u8_prof.jsonl"))
    ap.add_argument("--child", default="")
    ap.add_argument("--graph", default="")
    ap.add_argument("--dump", default="")
    ap.add_argument("--mode", default="load")
    a = ap.parse_args()
    if a.child == "build":
        return child_build(a)
    if a.child == "search":
        return child_search(a)

    try:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip().splitlines()
    except FileNotFoundError:
        card = ["nvidia-smi not found"]
    common = ["--n", str(a.n), "--nq", str(a.nq), "--efs", a.efs, "--reps", str(a.reps)]
    with tempfile.TemporaryDirectory() as tmp:
        graph = os.path.join(tmp, "u8.hnsw")
        lines = [{"what": "card", "nvidia_smi": card, "n": a.n, "nq": a.nq, "M": 16, "efConstruction": 200}]
        lines.append({"what": "build", **run_child(["--child", "build", "--graph", graph, *common], {}, "build")})
        exact = np.load(graph + ".exact.npy")
        runs = [("this", {}, "load")]
        if a.other_lib:
            runs.append(("other", {"NB200_LIB": a.other_lib}, "import"))
        answers = {}
        for rnd in range(a.rounds):
            for name, env, mode in runs:
                dump = os.path.join(tmp, f"{name}{rnd}.npz")
                recs = run_child(["--child", "search", "--graph", graph, "--dump", dump, "--mode", mode, *common],
                                 env, name)
                ans = np.load(dump)
                answers.setdefault(name, ans)
                row_bytes = 512 if name == "other" else 128
                for r in recs:
                    ids = ans[f"ids{r['ef']}"]
                    hits = sum(len(set(x.tolist()) & set(e.tolist())) for x, e in zip(ids, exact))
                    bpq = r["evals_per_q"] * row_bytes + r["expansions_per_q"] * 4 * MAXM0
                    r.update({"what": "search", "lib": name, "round": rnd, "recall10": hits / exact.size,
                              "row_bytes": row_bytes, "bytes_per_q": bpq,
                              "GBps": bpq * a.nq / (r["last_scan_ms"] * 1e-3) / 1e9})
                    lines.append(r)
        for evg in ([2, 4, 8] if a.evg_lib else []):
            dump = os.path.join(tmp, f"evg{evg}.npz")
            recs = run_child(["--child", "search", "--graph", graph, "--dump", dump, "--mode", "load", *common],
                             {"NB200_LIB": a.evg_lib, "NB200_HNSW_G": str(evg)}, f"evg {evg}")
            answers[f"evg{evg}"] = np.load(dump)
            for r in recs:
                r.update({"what": "evg", "evg": evg})
                lines.append(r)
        base = answers["this"]
        verdict = {"what": "identical"}
        for name, ans in answers.items():
            verdict[name] = all(np.array_equal(ans[key].view(np.int32), base[key].view(np.int32)) for key in base.files)
        lines.append(verdict)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    with open(a.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")
    for line in lines:
        print(json.dumps(line))
    if not all(v for k, v in verdict.items() if k != "what"):
        sys.exit("answers differ")


if __name__ == "__main__":
    main()
