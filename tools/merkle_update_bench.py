"""Incremental Merkle updates vs a full rebuild, one GPU, device-resident arity-4 trees.

    python tools/merkle_update_bench.py [--out profiles/r3_merkle_update.json] [--logn 11 13] [--calls 20]

For every tree (4^logn leaves) and every batch size k, two index patterns: `random` (uniform, with repeats) and
`range` (k consecutive leaves from a random start, append-like); k = 2^20 and 2^22 locate where a rebuild wins.  Per
point: ms per update (CUDA events on the engine's stream, warm-up first, --calls timed calls), the dirty digests
sum_l |unique(idx >> 2l)|, dirty digests/s, the full merkle_build of the same tree timed in the same run, and
update / rebuild.  After each tree's timed loop the updated tree is compared with a rebuild of its leaves.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K_VALUES = [1, 16, 256, 3552, 1 << 14, 1 << 16, 1 << 18, 1 << 20, 1 << 22]   # points with k > n_leaves are skipped


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [v.strip() for v in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                                   # the numbers are still valid, only unlabelled
        return {"error": str(e)}


def dirty_digests(idx, depth, log2_arity=2):
    u = np.unique(idx)
    total = 0
    for _ in range(depth):
        u = np.unique(u >> np.uint64(log2_arity))
        total += len(u)
    return int(total)


def time_calls(torch, fn, calls):
    """ms per call: CUDA events on the current (= engine) stream around `calls` back-to-back calls"""
    fn()
    fn()
    torch.cuda.current_stream().synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(calls):
        fn()
    t1.record()
    t1.synchronize()
    return t0.elapsed_time(t1) / calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--logn", type=int, nargs="+", default=[11, 13])
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.calls < 20:
        ap.error("--calls must be at least 20")
    import torch

    import poseidon252_b200 as pb
    from poseidon252_b200.scalar import random_limbs_fast

    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    eng = pb.Engine(0, stream=stream.cuda_stream)
    rng = np.random.default_rng(13)
    result = {"gpu": gpu_info(), "arity": 4, "calls_per_point": a.calls, "trees": []}
    for logn in a.logn:
        n = 4 ** logn
        leaves = torch.from_numpy(random_limbs_fast(rng, (n,)).reshape(n, 4).view(np.int64)).cuda()
        nodes = eng.merkle_build(leaves, arity=4)
        build_ms = time_calls(torch, lambda: eng.merkle_build(leaves, arity=4, out=nodes, async_=True), max(5, a.calls // 4))
        n_internal = int(nodes.shape[0])
        tree = {"logn": logn, "n_leaves": n, "depth": logn, "build_ms": build_ms, "build_digests": n_internal,
                "build_digests_per_s": n_internal / (build_ms * 1e-3), "points": []}
        for k in [k for k in K_VALUES if k <= n]:
            for pattern in ("random", "range"):
                if pattern == "random":
                    idx = rng.integers(0, n, size=k, dtype=np.uint64)
                else:
                    start = int(rng.integers(0, n - k + 1))
                    idx = np.arange(start, start + k, dtype=np.uint64)
                vals = random_limbs_fast(rng, (k,)).reshape(k, 4)
                d_idx = torch.from_numpy(idx.view(np.int64)).cuda()
                d_vals = torch.from_numpy(vals.view(np.int64)).cuda()
                ms = time_calls(torch, lambda: eng.merkle_update_batch(leaves, nodes, d_idx, d_vals, arity=4, async_=True),
                                a.calls)
                dd = dirty_digests(idx, logn)
                tree["points"].append({"k": k, "pattern": pattern, "update_ms": ms, "dirty_digests": dd,
                                       "dirty_digests_per_s": dd / (ms * 1e-3), "update_over_build": ms / build_ms})
                print(json.dumps({"logn": logn, **tree["points"][-1]}), flush=True)
        rebuilt = eng.merkle_build(leaves, arity=4)
        stream.synchronize()
        tree["parity_vs_rebuild"] = bool(torch.equal(rebuilt, nodes))
        # the largest k at which an update still beats the rebuild, per pattern
        for pattern in ("random", "range"):
            wins = [p["k"] for p in tree["points"] if p["pattern"] == pattern and p["update_ms"] < build_ms]
            tree["largest_k_faster_than_build_" + pattern] = max(wins) if wins else None
        result["trees"].append(tree)
        del leaves, nodes, rebuilt
        torch.cuda.empty_cache()
    eng.close()
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")
    ok = all(t["parity_vs_rebuild"] for t in result["trees"])
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
