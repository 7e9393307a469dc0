#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 Hades engine (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload W] [--dump-outputs DIR]

Workload (default `merkle4`, BASELINE.json configs[1]): one step = one batch of 2^20 independent
`Hash::digest(Domain::Merkle4, 4 scalars)` per GPU = 2^20 width-5 Hades permutations per GPU, on
synthetic uniform BlsScalars.  `value` = permutations/s of the whole job (all ranks), inputs resident
in HBM, timed with CUDA events on the launching stream, max over ranks.  `e2e` = the same metric through
the public API (`Hash.digest_batch`) with pinned HOST buffers: H2D + kernel + D2H inside the timed
region.  `--impl reference` times the reference's CPU algorithm (oracle/hades_ref.c, the faithful C
port: the Rust crate cannot be built here) on all host cores, on the SAME 2^20-digest batch per step, timing the
hashing call alone (inputs and tag are generated once, outside the loop).  N > 1 (torchrun): every rank hashes
its own shard, no collective on the data path (weak scaling).

The same JSON line also carries a `tree` block: the arity-4 Merkle tree build of BASELINE configs[3] scaled to
the GPUs present (4^14 leaves on 8 GPUs, 4^13 on 4, 4^12 on 2, 4^11 on 1), leaves sharded over the ranks, one NCCL
all-gather per level -- the only path north_star shards with a collective -- with its exposed-communication
time (full build vs a compute-only build with the gathers skipped), per-level kernel / all-gather device times,
and an in-run parity verdict against the CPU oracle (outside every timed region).

Other workloads (not the driver's headline; used for profiles/ and DESIGN.md numbers):
  --workload encrypt|decrypt   2^20 x encrypt/decrypt(L=2)  (configs[2])      --workload permute  raw 2^20 x 5 states
  --workload sweep     Domain::Other, EVERY in_len 1..256 at 2^18 items (configs[4]); per-length table in `sweep`
                       (--sweep-lens 1,2,4 to subsample)
  --workload tree      the tree build alone (--log4-leaves k)                  --workload convert  wire-format kernel

--dump-outputs DIR writes, after the timed steps, what the last timed step computed as DIR/<name>.npy, so that two
builds can be compared output for output on identical seeded inputs (see dump_outputs).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "hades_permutations_per_sec"
UNIT = "perm/s"
LOG2_BATCH = 20
BYTES_PER_PERM = 160          # Merkle4 digest: 4 x 32 B in + 32 B out (SURVEY.md 8d)
SM_COUNT = 148
TREE_LOG4 = {1: 11, 2: 12, 4: 13, 8: 14}
DUMP_ROWS = 1 << 16           # items kept per dumped array (4 MiB for Merkle4 digests)


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """nvidia-smi clocks / throttle reasons streamed (-lms) DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.15)                      # let the first samples arrive before the timed region
        except Exception:
            self.proc = None

    def stop(self):
        rows = []
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                self.proc.kill()
                out = ""
            for ln in out.splitlines():
                parts = [p.strip() for p in ln.split(",")]
                if len(parts) >= 7:
                    try:
                        float(parts[0])
                        rows.append(parts)
                    except ValueError:
                        pass
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = [float(r[0]) for r in rows]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[3 + k].lower().startswith("active") for r in rows)]
        return {"sm_mhz": statistics.median(sm), "sm_min_mhz": min(sm), "sm_max_mhz": float(rows[0][1]),
                "reasons": reasons, "power_w_max": max(float(r[2]) for r in rows), "samples": len(rows)}


def usable_cores():
    """Host threads this process may really use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """dram bytes per launch of the dominant kernel from the committed `ncu --set full` capture (newest round)."""
    for name in ("r2_ncu_summary.json", "r1_ncu_summary.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                v = json.load(f).get("merkle4_2p20", {}).get("dram_bytes_per_launch")
            if v:
                return v
        except Exception:
            pass
    return None


def dump_outputs(directory, arrays, rank, world):
    """Writes each array (numpy or torch, first axis = items) as <directory>/<name>.npy in float64, one row per item.
    Batches larger than DUMP_ROWS items keep a fixed seeded sample of DUMP_ROWS rows in item order.  Every 64-bit word
    is split into its 32-bit halves, low half first, so that each value is exact in float64.  With more than one rank,
    each rank writes <name>_rank<r>.npy."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    suffix = "" if world == 1 else "_rank%d" % rank
    for name, a in arrays.items():
        a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
        a = np.ascontiguousarray(a.reshape(a.shape[0], -1))
        if a.shape[0] > DUMP_ROWS:
            a = a[np.sort(np.random.default_rng(0xD0).choice(a.shape[0], DUMP_ROWS, replace=False))]
        if a.dtype.itemsize == 8:
            a = a.view(np.uint32)
        np.save(os.path.join(directory, name + suffix + ".npy"), a.astype(np.float64))


def workload_config(log2_batch, world):
    """`config` of the headline workload -- built by ONE function so that the GPU arm and the reference arm print the
    identical object (the driver compares them)."""
    n = 1 << log2_batch
    return {"workload": "batch 2^%d Domain::Merkle4 digests (4 scalars -> 1) per GPU" % log2_batch,
            "per_gpu_batch": n,
            "l2": "inputs rotate over 4 distinct %d MiB device buffers (each > L2)" % (n * 128 >> 20),
            "parallelism": "dp%d, no collective on the data path" % world}


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm on the host cores (oracle C port; test infrastructure)
# ---------------------------------------------------------------------------------------------------------
class CpuArm:
    """Merkle4-shaped digests with the dense reference algorithm (oracle/hades_ref.c).  Inputs, tag and the output
    buffer are created ONCE here; run() times nothing but the hashing call."""

    def __init__(self, n_items, in_len=4, seed=123):
        import numpy as np
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import c_oracle
        import hades_oracle as o
        from poseidon252_b200.scalar import random_limbs_fast, to_mont
        self.c_oracle, self.in_len, self.n = c_oracle, in_len, n_items
        self.data = random_limbs_fast(np.random.default_rng(seed), (n_items, in_len))
        self.out = np.zeros((n_items, 1, 4), dtype=np.uint64)
        self.tag = to_mont(o.hash_to_scalar(o.tag_input([o.Absorb(in_len), o.Squeeze(1)], o.Domain.Merkle4)))
        c_oracle.digest(self.tag, self.data[:64], in_len, 1)          # load + initialise the library

    def run(self, threads, n=None):
        """seconds spent inside oracle_digest[_mt] for the first n items"""
        n = self.n if n is None else min(n, self.n)
        t0 = time.perf_counter()
        self.c_oracle.digest(self.tag, self.data[:n], self.in_len, 1, threads=threads, out=self.out[:n])
        return time.perf_counter() - t0


def cpu_baseline_block(target_seconds=10.0):
    threads = usable_cores()
    arm = CpuArm(1 << 22)
    probe_n = min(arm.n, 4096 * threads)
    arm.run(threads, probe_n)
    rate = probe_n / arm.run(threads, probe_n)
    n = int(min(arm.n, max(probe_n, rate * target_seconds)))
    dt = arm.run(threads, n)
    # criterion's `hash 4 BlsScalar` shape (benches/hash.rs:68-72): one digest at a time on one thread
    n1 = 4096
    arm.run(1, n1)
    dt1 = arm.run(1, n1)
    return {"value": n / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "%d Merkle4 digests (1 permutation each) of the dense reference algorithm "
                      "(oracle/hades_ref.c, 4x64-bit Montgomery), %d pthreads, %.1f s; hashing call timed alone" % (n, threads, dt),
            "single_thread": {"value": n1 / dt1, "unit": UNIT, "us_per_digest": dt1 / n1 * 1e6,
                              "sample": "%d digests, 1 thread (criterion `hash 4 BlsScalar` shape, benches/hash.rs:68-72)" % n1}}


def run_reference_arm(args, rank, world, emit):
    if rank != 0:
        return
    threads = usable_cores()
    n = 1 << args.log2_batch
    arm = CpuArm(n)
    probe_n = min(n, 4096 * threads)
    arm.run(threads, probe_n)
    rate = probe_n / arm.run(threads, probe_n)
    # the full 2^20-digest batch per step; only a host so slow that the run would exceed ~15 min gets a bounded sample
    per_step, bounded = n, False
    if n / rate * (args.steps + args.warmup) > 900.0:
        per_step, bounded = int(max(probe_n, rate * 900.0 / (args.steps + args.warmup))), True
    for _ in range(args.warmup):
        arm.run(threads, per_step)
    dts = [arm.run(threads, per_step) for _ in range(args.steps)]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"digests": arm.out[:per_step]}, rank, 1)
    total = sum(dts)
    value = per_step * args.steps / total
    sample = "%d digests per step x %d steps, %d pthreads; hashing call timed alone (inputs/tag generated once, outside)" % (
        per_step, args.steps, threads)
    if bounded:
        sample += "; BOUNDED sample of the 2^%d batch (slow host)" % args.log2_batch
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64 limbs (255-bit modular integer)", "data": "synthetic",
            "config": workload_config(args.log2_batch, world),
            "algorithm": "reference dense Hades (src/hades/permutation/scalar.rs:39-64), C port oracle/hades_ref.c "
                         "(the Rust crate cannot be built in this image)",
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ---------------------------------------------------------------------------------------------------------
# Tree block: arity-4 Merkle build, leaves sharded over the ranks, one NCCL all-gather per level
# ---------------------------------------------------------------------------------------------------------
def device_random_scalars(torch, n, seed):
    """(n, 4) int64 CUDA tensor of valid BlsScalar.0 limbs (top limb below p's top limb), generated on the device."""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    a = torch.randint(-(1 << 63), (1 << 63) - 1, (n, 4), dtype=torch.int64, device="cuda", generator=g)
    a[:, 3] = torch.randint(0, 0x73EDA753299D7D48, (n,), dtype=torch.int64, device="cuda", generator=g)
    return a


def tree_block(eng, torch, dist, rank, world, stream, k, builds=3, paths=64):
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import c_oracle
    import hades_oracle as o
    from poseidon252_b200 import merkle
    from poseidon252_b200.scalar import to_mont

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    tag = to_mont(o.hash_to_scalar(o.tag_input([o.Absorb(4), o.Squeeze(1)], o.Domain.Merkle4)))
    parity = {}
    with torch.cuda.stream(stream):
        # ---- parity (a): a 4^8 tree through the SAME distributed path equals the single-GPU build and the oracle ----
        small = 4 ** 8
        sh = small // world
        s_leaves = device_random_scalars(torch, sh, 1000 + rank)
        s_nodes = eng.merkle4_build_dist(s_leaves, small)
        stream.synchronize()
        if dist is not None:
            parts = [torch.empty_like(s_leaves) for _ in range(world)]
            dist.all_gather(parts, s_leaves)
            all_leaves = torch.cat(parts, dim=0)
        else:
            all_leaves = s_leaves
        single = eng.merkle4_build(all_leaves)
        stream.synchronize()
        ok_a = bool(torch.equal(single, s_nodes))
        if rank == 0:
            cur = all_leaves.cpu().numpy().view(np.uint64)
            lv = []
            while cur.shape[0] > 1:
                cur = c_oracle.digest(tag, cur.reshape(-1, 4, 4), 4, 1, threads=usable_cores()).reshape(-1, 4)
                lv.append(cur)
            ok_a = ok_a and bool(np.array_equal(np.concatenate(lv, axis=0), s_nodes.cpu().numpy().view(np.uint64)))
        parity["small_tree_4p8_equals_single_gpu_and_oracle"] = ok_a
        del s_leaves, s_nodes, all_leaves, single

        # ---- the big tree ----
        n_leaves = 4 ** k
        shard = n_leaves // world
        n_internal, n_levels = eng.tree_nodes(n_leaves)
        leaves = device_random_scalars(torch, shard, 77 + rank)
        nodes = torch.empty((n_internal, 4), dtype=torch.int64, device="cuda")
        for _ in range(2):
            eng.merkle4_build_dist(leaves, n_leaves, out=nodes, async_=True)
    barrier()

    def timed(n_builds, **kw):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(n_builds + 1)]
        with torch.cuda.stream(stream):
            ev[0].record(stream)
            for i in range(n_builds):
                eng.merkle4_build_dist(leaves, n_leaves, out=nodes, async_=True, **kw)
                ev[i + 1].record(stream)
        stream.synchronize()
        barrier()
        return max_over_ranks(ev[0].elapsed_time(ev[-1]) / n_builds)

    ms_full = timed(builds)

    # ---- parity (b): `paths` random leaf -> root paths of the big tree recomputed with the CPU oracle ----
    offs = merkle.level_offsets(n_leaves)
    rng = np.random.default_rng(4242 + rank)
    idx = rng.integers(0, shard, size=paths)
    ok_b = True
    g = idx // 4
    group = leaves[torch.from_numpy(np.stack([4 * g + q for q in range(4)], axis=1)).cuda()]      # (paths, 4, 4) own leaves
    gidx = (rank * shard + idx) // 4                                                            # global node index, level 0
    for lvl, (off, size) in enumerate(offs):
        want = c_oracle.digest(tag, group.cpu().numpy().view(np.uint64), 4, 1).reshape(-1, 4)
        got = nodes[torch.from_numpy(off + gidx).cuda()].cpu().numpy().view(np.uint64)
        ok_b = ok_b and bool(np.array_equal(want, got))
        if size == 1:
            break
        g = gidx // 4
        group = nodes[torch.from_numpy(np.stack([off + 4 * g + q for q in range(4)], axis=1)).cuda()]
        gidx = g
    if dist is not None:
        t = torch.tensor([1.0 if (ok_b and ok_a) else 0.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        all_ok = bool(t.item() == 1.0)
    else:
        all_ok = ok_a and ok_b
    parity["%d_random_leaf_to_root_paths_per_rank_vs_oracle" % paths] = ok_b

    # ---- per-level device times (one build with events), then the compute-only run ----
    with torch.cuda.stream(stream):
        eng.merkle4_build_dist(leaves, n_leaves, out=nodes, async_=True, timing=True)
    stream.synchronize()
    levels, total_timed = eng.tree_level_timings()
    barrier()
    ms_compute = timed(builds, no_gather=True) if world > 1 else ms_full
    per_level = []
    for l, t in enumerate(levels):
        row = {"level": l, "nodes": t["nodes"], "my_nodes": t["my_nodes"], "kernel_ms": round(t["kernel_ms"], 4)}
        if t["gather_bytes"]:
            row.update(gather_ms=round(t["gather_ms"], 4), gather_MiB=t["gather_bytes"] >> 20,
                       gather_GBps=round(t["gather_bytes"] * (world - 1) / world / (t["gather_ms"] * 1e-3) / 1e9, 1) if t["gather_ms"] > 0 else None)
        per_level.append(row)
    small_levels = [r for r in per_level if r["nodes"] < 740 * 128]
    exposed = max(0.0, ms_full - ms_compute)
    worst = max((r for r in per_level if "gather_ms" in r), key=lambda r: r["gather_ms"], default=None)
    limiting = ("levels with < 1 wave of blocks are latency-bound: %d levels, %.2f ms of kernels" %
                (len(small_levels), sum(r["kernel_ms"] for r in small_levels)))
    if worst is not None:
        limiting += "; largest collective = level %d all-gather (%d MiB, %.2f ms), exposed all-gather total %.2f ms" % (
            worst["level"], worst["gather_MiB"], worst["gather_ms"], exposed)
    return {"workload": "arity-4 Merkle tree, 4^%d = 2^%d leaves over %d GPU(s), %d levels, one NCCL all-gather per level"
                        % (k, 2 * k, world, n_levels),
            "leaves_log4": k, "digests": n_internal, "builds_timed": builds,
            "ms_per_tree": ms_full, "value": n_internal / (ms_full * 1e-3), "unit": UNIT, "scaling": "strong",
            "compute_only_ms": ms_compute, "exposed_allgather_ms": exposed,
            "gathered_MiB_per_rank": sum(t["gather_bytes"] for t in levels) >> 20,
            "timed_build_ms_rank0": total_timed, "per_level_rank0": per_level, "limiting": limiting,
            "parity": "ok" if all_ok else "MISMATCH", "parity_checks": parity}


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 40; 2 for --workload sweep: one step = 2.2e9 permutations)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="merkle4", choices=["merkle4", "encrypt", "decrypt", "permute", "sweep", "tree", "convert"])
    ap.add_argument("--log2-batch", type=int, default=LOG2_BATCH)
    ap.add_argument("--log4-leaves", type=int, default=0, help="tree: 4^k leaves in the whole job (14 = BASELINE configs[3])")
    ap.add_argument("--sweep-lens", default="", help="sweep: comma-separated input lengths (default: every length 1..256)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-tree", action="store_true", help="merkle4: skip the tree block")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 2 if args.workload == "sweep" else 40
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.workload == "tree" and args.impl == "b200":
        ap.error("--dump-outputs is not supported with --workload tree")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)

    # Exactly ONE line may reach stdout (the JSON); native libraries (e.g. NCCL's version banner) write to
    # fd 1 too, so fd 1 is pointed at stderr for the duration of the run and the JSON goes to the saved fd.
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    def emit(obj):
        real_stdout.write(json.dumps(obj) + "\n")
        real_stdout.flush()

    if args.impl == "reference":
        run_reference_arm(args, rank, world, emit)
        return

    import numpy as np
    import torch
    import poseidon252_b200 as pb
    from poseidon252_b200.scalar import random_limbs_fast

    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    stream = torch.cuda.Stream()
    eng = pb.Engine(local, stream=stream.cuda_stream)
    tree_skip = None
    if dist is not None and args.workload in ("merkle4", "tree") and not (args.workload == "merkle4" and args.no_tree):
        # the library's own NCCL communicator (bound with dlopen to the NCCL copy torch already loaded); if any rank
        # cannot set it up, every rank skips the tree block instead of losing the headline
        ok = 1.0
        try:
            box = [eng.dist_unique_id() if rank == 0 else bytes(128)]
        except Exception as exc:
            box, ok, tree_skip = [bytes(128)], 0.0, repr(exc)
        dist.broadcast_object_list(box, src=0)
        flag = torch.tensor([ok], dtype=torch.float64, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if flag.item() == 1.0:
            try:
                eng.dist_init(box[0], rank, world)
            except Exception as exc:
                ok, tree_skip = 0.0, repr(exc)
            flag = torch.tensor([ok], dtype=torch.float64, device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if flag.item() != 1.0:
            tree_skip = tree_skip or "another rank could not initialise the tree communicator"
            if args.workload == "tree":
                raise RuntimeError(tree_skip)
    n = 1 << args.log2_batch
    rng = np.random.default_rng(0xC10D + rank)          # benches/hash.rs:53 seed, per-rank stream

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    extra = {}
    config = None
    per_launch_events = False
    # ---- workload set-up: step(i) enqueues one batch on `stream`; returns perms per step ----------------
    if args.workload == "merkle4":
        nbuf = 4                                          # rotate over 4 x 128 MiB inputs (> 126 MB L2)
        with torch.cuda.stream(stream):
            ins = [torch.from_numpy(random_limbs_fast(rng, (n, 4)).view(np.int64)).cuda() for _ in range(nbuf)]
            out = torch.empty((n, 1, 4), dtype=torch.int64, device="cuda")
        perms_per_step, bytes_per_step = n, n * BYTES_PER_PERM
        step = lambda i: pb.Hash.digest_batch(pb.Domain.Merkle4, ins[i % nbuf], engine=eng, out=out, async_=True)
        outputs = lambda: {"digests": out}
        config = workload_config(args.log2_batch, world)
    elif args.workload == "permute":
        with torch.cuda.stream(stream):
            st = torch.from_numpy(random_limbs_fast(rng, (n, 5)).view(np.int64)).cuda()
        perms_per_step, bytes_per_step = n, n * 320
        step = lambda i: eng.permute_batch_inplace(st, async_=True)
        outputs = lambda: {"states": st}
        workload, l2_note = "raw permute_batch of 2^%d x 5 states in place" % args.log2_batch, "160 MiB state array > L2"
    elif args.workload == "encrypt":
        with torch.cuda.stream(stream):
            msg = torch.from_numpy(random_limbs_fast(rng, (n, 2)).view(np.int64)).cuda()
            sec = torch.from_numpy(random_limbs_fast(rng, (n, 2)).view(np.int64)).cuda()
            non = torch.from_numpy(random_limbs_fast(rng, (n,)).view(np.int64)).cuda()
            cip = torch.empty((n, 3, 4), dtype=torch.int64, device="cuda")
        perms_per_step, bytes_per_step = 2 * n, n * 256
        step = lambda i: pb.encrypt_batch(msg, sec, non, engine=eng, out=cip, async_=True)
        outputs = lambda: {"ciphertexts": cip}
        workload, l2_note = "encrypt_batch 2^%d messages, L=2 (benches/encrypt.rs:17)" % args.log2_batch, "256 MiB touched per step > L2"
    elif args.workload == "decrypt":
        with torch.cuda.stream(stream):
            msg = torch.from_numpy(random_limbs_fast(rng, (n, 2)).view(np.int64)).cuda()
            sec = torch.from_numpy(random_limbs_fast(rng, (n, 2)).view(np.int64)).cuda()
            non = torch.from_numpy(random_limbs_fast(rng, (n,)).view(np.int64)).cuda()
        cip = pb.encrypt_batch(msg, sec, non, engine=eng)
        eng.sync()
        perms_per_step, bytes_per_step = 2 * n, n * (192 + 64 + 1)
        ok_holder = {}

        def step(i):
            ok_holder["m"], ok_holder["ok"] = pb.decrypt_batch(cip, sec, non, engine=eng, async_=True)
        outputs = lambda: {"messages": ok_holder["m"], "ok": ok_holder["ok"]}
        workload, l2_note = "decrypt_batch 2^%d ciphers, L=2 (benches/decrypt.rs:17)" % args.log2_batch, "257 MiB touched per step > L2"
    elif args.workload == "sweep":
        n = 1 << 18
        lens = [int(v) for v in args.sweep_lens.split(",")] if args.sweep_lens else list(range(1, 257))
        with torch.cuda.stream(stream):
            # ONE 2 GiB buffer of valid scalars; length L reads its first n*L scalars as (n, L, 4)
            flat = torch.from_numpy(random_limbs_fast(rng, (n * max(lens),)).view(np.int64)).cuda()
            out = torch.empty((n, 1, 4), dtype=torch.int64, device="cuda")
        views = {L: flat[: n * L].view(n, L, 4) for L in lens}
        perms_per_step = sum(n * ((L + 3) // 4) for L in lens)
        bytes_per_step = sum(n * (32 * L + 32) for L in lens)
        sweep_events = []

        def step(i):
            evs = [torch.cuda.Event(enable_timing=True)]
            evs[0].record(stream)
            for L in lens:
                pb.Hash.digest_batch(pb.Domain.Other, views[L], engine=eng, out=out, async_=True)
                e = torch.cuda.Event(enable_timing=True)
                e.record(stream)
                evs.append(e)
            sweep_events.append(evs)
        outputs = lambda: {"digests_in_len%d" % lens[-1]: out}        # `out` holds the step's last length
        workload = "sponge sweep Domain::Other, every in_len in [%d, %d] (%d lengths), batch 2^18 per length per GPU" % (
            min(lens), max(lens), len(lens))
        l2_note = "length L reads the first 2^18*L scalars of one %d MiB buffer (> L2 for L >= 16)" % (n * max(lens) * 32 >> 20)
    elif args.workload == "convert":
        n = 1 << 25                                       # 1 GiB of scalars in, 1 GiB of bytes out
        with torch.cuda.stream(stream):
            sc = torch.from_numpy(random_limbs_fast(rng, (n,)).view(np.int64)).cuda()
            ob = torch.empty((n, 4), dtype=torch.int64, device="cuda")
        perms_per_step, bytes_per_step = n, n * 64       # "perms" here = scalars converted (no permutation)
        lib, ctx = eng._lib, eng._ctx
        step = lambda i: eng._check(lib.p252_scalars_to_bytes(ctx, sc.data_ptr(), n, ob.data_ptr(), 3))
        outputs = lambda: {"bytes": ob}
        workload, l2_note = "to_bytes of 2^25 scalars (wire-format kernel, the one HBM-bound kernel); value = scalars/s", "1 GiB in + 1 GiB out per step"
    else:  # tree alone
        k = args.log4_leaves or TREE_LOG4.get(world, 12)
        blk = tree_block(eng, torch, dist, rank, world, stream, k, builds=max(3, min(args.steps, 10)))
        if rank == 0:
            clocks = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
            line = {"metric": METRIC, "value": blk["value"], "unit": UNIT, "n_gpus": world, "steps": blk["builds_timed"],
                    "warmup": 2, "ms_per_step": blk["ms_per_tree"], "higher_is_better": True, "scaling": "strong",
                    "vs_baseline": None, "dtype": "u32 limbs (255-bit modular integer, IMAD.WIDE carry chains)",
                    "data": "synthetic", "config": {"workload": blk["workload"]}, "clocks": clocks,
                    "gpu_launches": blk["leaves_log4"] * blk["builds_timed"], "tree": blk}
            emit(line)
        if dist is not None:
            dist.destroy_process_group()
        return
    if config is None:
        config = {"workload": workload, "per_gpu_batch": perms_per_step, "l2": l2_note,
                  "parallelism": "dp%d, no collective on the data path" % world}

    stream.synchronize()
    with torch.cuda.stream(stream):
        for i in range(args.warmup):
            step(i)
    barrier()
    if args.workload == "sweep":
        sweep_events.clear()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = eng.launch_count
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    with torch.cuda.stream(stream):
        ev[0].record(stream)
        for i in range(args.steps):
            step(i)
            ev[i + 1].record(stream)
    stream.synchronize()
    barrier()
    clocks = sampler.stop()
    launches = eng.launch_count - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs(), rank, world)
    total_ms = ev[0].elapsed_time(ev[-1])
    per_step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    if dist is not None:
        t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    job_perms = perms_per_step * args.steps * world
    value = job_perms / (total_ms * 1e-3)
    if args.workload == "sweep":
        # per-length device time (median over the timed steps) -> perm/s per input length
        table = []
        for j, L in enumerate(lens):
            ms = statistics.median(evs[j].elapsed_time(evs[j + 1]) for evs in sweep_events)
            table.append({"in_len": L, "perms_per_item": (L + 3) // 4, "ms": round(ms, 4),
                          "perm_per_s": n * ((L + 3) // 4) / (ms * 1e-3)})
        extra["sweep"] = table

    # ---- e2e: public API, pinned host buffers, H2D + kernel + D2H inside the timed region ---------------
    e2e = None
    if args.workload == "merkle4":
        h_in = torch.from_numpy(random_limbs_fast(rng, (n, 4)).view(np.int64)).pin_memory()
        h_out = torch.empty((n, 1, 4), dtype=torch.int64).pin_memory()
        a_in, a_out = h_in.numpy().view(np.uint64), h_out.numpy().view(np.uint64)
        e_steps = max(3, min(args.steps, 10))
        for _ in range(2):
            pb.Hash.digest_batch(pb.Domain.Merkle4, a_in, engine=eng, out=a_out)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        t0 = time.perf_counter()
        for _ in range(e_steps):
            pb.Hash.digest_batch(pb.Domain.Merkle4, a_in, engine=eng, out=a_out)      # synchronous HOST call
        e1.record(stream)
        stream.synchronize()
        wall_ms = (time.perf_counter() - t0) * 1e3
        e_ms = max(e0.elapsed_time(e1), wall_ms)
        if dist is not None:
            t = torch.tensor([e_ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e_ms = float(t.item())
        e2e = {"value": n * e_steps * world / (e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": n * 128,
               "d2h_bytes_per_step": n * 32, "steps": e_steps, "ms_per_step": e_ms / e_steps,
               "api": "poseidon252_b200.Hash.digest_batch(Domain.Merkle4, pinned host array) -> p252_hash_batch(P252_MEM_HOST)"}

    # ---- tree block (all ranks take part; outside the headline's timed region) ----------------------------------
    tree = None
    if args.workload == "merkle4" and not args.no_tree and tree_skip is not None:
        tree = {"error": "tree block skipped: " + tree_skip}
    elif args.workload == "merkle4" and not args.no_tree:
        try:
            del ins
            torch.cuda.empty_cache()
            tree = tree_block(eng, torch, dist, rank, world, stream, args.log4_leaves or TREE_LOG4.get(world, 12))
        except Exception as exc:  # never hide the headline because of the additional block
            tree = {"error": repr(exc)}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    peak, peak_src = measured_peaks()
    launches_per_step = max(1, launches // args.steps)
    launch_ms = statistics.mean(per_step_ms) / launches_per_step
    achieved = bytes_per_step / launches_per_step / (launch_ms * 1e-3) / 1e9
    info = eng.kernel_info()
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    # Integer-multiplier roofline, computed from THIS run: the multiplier instructions one permutation issues (counted
    # by the PTX generator, exported by the library) x the measured permutation rate, against one IMAD.WIDE per 4
    # cycles per SM sub-partition (measured: tools/microbench/pipe_table.cu) at the SM clock sampled during the run.
    wide_rate = info["wide_mul_per_permutation"] * (value / world) / 32.0          # warp instructions / s / GPU
    wide_peak = SM_COUNT * 4 * sm_mhz * 1e6 / 4.0
    imad = {"bound": "imad", "achieved": wide_rate / 1e9, "peak": wide_peak / 1e9, "unit": "G warp-IMAD.WIDE/s",
            "frac": wide_rate / wide_peak, "wide_mul_per_permutation": info["wide_mul_per_permutation"],
            "dfma_per_permutation": info["dfma_per_permutation"], "sm_mhz": sm_mhz,
            "peak_source": "148 SMs x 4 sub-partitions x SM clock / 4 cycles per IMAD.WIDE (B200 measurement, "
                           "profiles/r2_pipe_table.log); clock = median nvidia-smi sample of this run",
            "note": "achieved = multiplier instructions per permutation (library: p252_get_kernel_info) x measured perm/s / 32"}
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic(), "peak_source": peak_src,
                "kernel": "k_sponge_digest" if args.workload in ("merkle4", "sweep") else
                          ("k_crypt<false>" if args.workload == "encrypt" else "k_crypt<true>" if args.workload == "decrypt" else
                           ("k_convert<false>" if args.workload == "convert" else "k_permute<false>")),
                "algorithmic_bytes_per_launch": bytes_per_step // launches_per_step,
                "launch_ms": launch_ms,
                "note": "the path is integer-multiplier bound (~10^3 integer ops per byte), not HBM bound: see `imad`",
                "imad": imad if args.workload != "convert" else None}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32 limbs (255-bit modular integer, IMAD.WIDE carry chains)", "data": "synthetic",
            "config": config, "clocks": clocks, "gpu_launches": launches, "roofline": roofline, "target_perm_per_s_1gpu": 1e8}
    line.update(extra)
    if e2e is not None:
        line["e2e"] = e2e
    if tree is not None:
        line["tree"] = tree
    if world == 1 and not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = cpu_baseline_block()
        except Exception as exc:  # the oracle is only a reported baseline; never hide the GPU number
            line["cpu_baseline"] = {"error": repr(exc)}
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
