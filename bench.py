#!/usr/bin/env python
"""bench.py -- BASELINE.json's headline metric on its configs[1] workload.

Workload "C2": FMT* precompute in the 2-D unit square, N = 1M synthetic uniform samples per
GPU, obstacle set ISRR_2H: one step = uniform-grid build + r-ball neighbour table (K1+K2) +
point validity (K6) + validity of every stored edge (K7: column classify + per-edge kernel).  metric = collision-checked edges/s
(the NN-queries/s figure of the same step is reported beside it).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

N > 1: launched by torch.distributed.run, one rank per GPU.  The headline line is WEAK scaling -- the
sample set grows to N x 1M (replicated on every GPU, stripe order), rank g owns the query columns
[g*1M, (g+1)*1M); the per-rank CSC shards concatenate, and every step ends with the one exchange the host
planner needs: the shard column lengths and edge-validity words of every rank on every rank (direct peer
stores over NVLink + a device flag barrier, csrc/xchg.cu; NCCL all-gather as the fallback).  The same line
carries, as sub-objects, the two multi-GPU configurations BASELINE.json names literally:
  "strong_scaling" -- N = 1M samples IN TOTAL sharded over the N GPUs (configs[1]),
  "mc"             -- 1e8 importance-sampled rollouts sharded by rollout id + all-reduce (configs[4]),
and at N = 1 a "secondary" block with configs C3 / C4 / C5 (own roofline + cpu_baseline each).
After the timed region every rank count checks the tables it just timed against the CPU oracle on
sampled column windows ("parity_checked": columns) -- including the GATHERED global colptr / validity bits.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SAMPLES_PER_GPU = 1_000_000
SEED = 20240602
METRIC = "collision_checked_edges_per_sec"
UNIT = "edges/s"


def workload_name(n_total, r):
    """the ONE workload string both arms print (the driver compares the two config blocks)"""
    return "C2: FMT* 2-D unit square, ISRR_2H, N=%d uniform samples (%d query columns per GPU), r=%.7f" % (
        n_total, SAMPLES_PER_GPU, r)


def fill_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of rball_fill<2, U> on this workload, from the
    committed `ncu --set full` capture of the newest round (profiles/rN/traffic.json, scripts/ncu_traffic.py);
    None when no capture is committed.  Measured under the profiler, so it is traffic only, never a time."""
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*", "traffic.json")), reverse=True):
        try:
            with open(path) as f:
                t = json.load(f)
        except (OSError, ValueError):
            continue
        for k, v in t.items():
            if k.startswith("rball_fill<2"):
                return v["dram_bytes_per_launch"]
    return None


def morton_order(V, bits=16):
    """argsort of 2-D points along a Z-order curve (host, numpy) -- for the auxiliary 'renumbered samples' figure"""
    q = np.minimum((V * (1 << bits)).astype(np.uint64), (1 << bits) - 1)

    def spread(x):
        x = (x | (x << 16)) & 0x0000FFFF0000FFFF
        x = (x | (x << 8)) & 0x00FF00FF00FF00FF
        x = (x | (x << 4)) & 0x0F0F0F0F0F0F0F0F
        x = (x | (x << 2)) & 0x3333333333333333
        x = (x | (x << 1)) & 0x5555555555555555
        return x
    return np.argsort(spread(q[:, 0]) | (spread(q[:, 1]) << 1), kind="stable")


def fmt_radius(N, d, rm=1.0, vol=1.0):
    import math
    return rm * 2 * (1 / d * vol / (math.pi ** (d / 2) / math.gamma(d / 2 + 1)) * math.log(N) / N) ** (1 / d)


def make_samples(n_total, stripe_order):
    V = np.random.Generator(np.random.PCG64(SEED)).random((n_total, 2))
    if stripe_order:
        # stripe order: each rank's query range is then a spatial stripe and its grid covers only the
        # stripe + r (FMT* is invariant to the order of i.i.d. samples; N = 1 keeps the raw order)
        V = V[np.argsort(V[:, 0], kind="stable")]
    return np.ascontiguousarray(V)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (pynvml, 2 ms period: the region is tens of ms)."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _sample(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
        }
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for k, bit in names.items():
                if mask & bit:
                    self.reasons.add(k)
        except Exception:
            pass

    def _loop(self):
        while not self._stop.is_set():
            self._sample()
            time.sleep(0.002)

    def start(self):
        if self.nv:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------
def oracle_step(orc, V, r, q0, q1, tree, O, So):
    """The reference's CPU path for columns [q0, q1): per-query kd-tree inball (sorted sparse
    column, nearneighbors.jl:179-183) + is_free_state for those samples + is_free_motion for
    every stored edge (robots2D.jl:13-14)."""
    colptr, rowval, nzval = tree.rball(r, q0, q1)
    orc.states_free(O, So, V[q0:q1])
    orc.edges_free_csc(O, So, V, colptr, rowval, q0)
    return len(rowval)


def run_oracle(V, r, q0, q1, threads, tree=None):
    """Time the oracle on columns [q0,q1) with `threads` host threads (ctypes drops the GIL).
    The kd-tree build (geometric.jl:14) is part of the timed path, done once, single-threaded
    as in the reference; pass `tree=(tree, t_build)` to reuse one."""
    from oracle import oracle as orc
    import fixtures as fx
    O = orc.Obstacles2D(fx.ISRR_2H)
    So = orc.StateSpace([0, 0], [1, 1])
    if tree is None:
        t0 = time.perf_counter()
        tree = orc.KDTree(V)
        t_build = time.perf_counter() - t0
    else:
        tree, t_build = tree
    bounds = np.linspace(q0, q1, threads + 1).astype(np.int64)
    edges = [0] * threads

    def work(i):
        edges[i] = oracle_step(orc, V, r, int(bounds[i]), int(bounds[i + 1]), tree, O, So)

    t0 = time.perf_counter()
    if threads == 1:
        work(0)
    else:
        ts = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
        [t.start() for t in ts]
        [t.join() for t in ts]
    t_q = time.perf_counter() - t0
    return sum(edges), t_build, t_q


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def reference_arm(args, rank, world):
    """--impl reference: the oracle port of the reference's CPU path, all host threads, rank 0 only."""
    if rank != 0:
        return
    n_total = SAMPLES_PER_GPU * world
    V = make_samples(n_total, world > 1)
    r = fmt_radius(n_total, 2)
    threads = host_threads()
    # bounded sample: a contiguous block of query columns, sized from one probe so that
    # (warmup + steps) stays within ~2 minutes
    probe = 20_000
    from oracle import oracle as orc
    t0 = time.perf_counter()
    tree = (orc.KDTree(V), 0.0)
    tree = (tree[0], time.perf_counter() - t0)
    _, tb, tq = run_oracle(V, r, 0, probe, threads, tree)
    per_col = tq / probe
    budget = 100.0 / max(1, args.steps + args.warmup)
    ncols = int(min(SAMPLES_PER_GPU * world, max(probe, budget / per_col)))
    times, edges = [], 0
    for it in range(args.warmup + args.steps):
        e, tb, tq = run_oracle(V, r, 0, ncols, threads, tree)
        # the tree build is amortised over the full sample set in the real workload: charge the
        # sample its proportional share
        t = tq + tb * (ncols / n_total)
        if it >= args.warmup:
            times.append(t)
            edges = e
    ms = 1e3 * float(np.mean(times))
    value = edges / (ms / 1e3)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(n_total, r)},
        "reference_sample_columns": ncols,
        "nn_queries_per_sec": ncols / (ms / 1e3),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "%d of %d query columns (kd-tree inball + point + edge checks), tree build charged pro rata; "
                                   "the reference itself is single-threaded -- this arm uses every host thread"
                                   % (ncols, n_total)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
class Job:
    """One sharded C2 precompute: sample set on the device, checker, exchange, and the step function."""

    def __init__(self, mp, V, q0, q1, world, tag):
        from mpb200 import sharding
        import torch
        import torch.distributed as dist
        self.mp, self.V, self.q0, self.q1, self.world = mp, V, q0, q1, world
        self.r = fmt_radius(len(V), 2)
        self.CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
        self.SS = mp.UnitHypercube(2)
        self.CC.handle()
        self.NN = mp.MetricNN(V)
        self.NN.set_query_range(q0, q1)
        self.NN.handle()  # inputs resident in HBM before the timed region
        self.exchange = None
        self.exchange_kind = None
        if world > 1:
            nnz0 = self.NN.build_table(self.r)
            self.exchange = sharding.make_exchange(q1 - q0, (nnz0 * 21 // 20 + 63) // 64 + 2)
            self.exchange_kind = "peer-stores" if isinstance(self.exchange, sharding.PeerExchange) else "nccl-allgather"
            if self.exchange_kind == "peer-stores":
                self.exchange.attach(self.NN.table)   # column lengths leave right after the count scan, under the fill
        self.nnz = 0
        self.pushes = 0
        self.exchange_ms = []
        self.lib = mp.load()

    def step(self):
        # the three calls of a planning step, issued back to back: only build_table waits (for nnz, once,
        # between count and fill); the validity calls enqueue their kernels and return
        NN = self.NN
        NN.points_free(self.CC, self.SS, fetch=False)           # K6
        self.nnz = NN.build_table(self.r)                       # K1 + K2
        NN.edges_free(NN.table, self.CC, self.SS, fetch=False, count=False)  # K7
        if self.exchange is not None:
            if self.exchange_kind == "peer-stores" and self.pushes > 0:
                # device time of the PREVIOUS push + barrier: complete by now (this step's nnz read-back is ordered
                # behind it), so reading it here never stalls the host; reading it at the end of its own step would
                # make every rank's host wait for the barrier before it may enqueue the next step
                self.exchange_ms.append(self.lib.mpb200_last_ms_of(3, 1))
            self.exchange.run(NN.table)          # column lengths + validity words of every rank -> every rank
            self.pushes += 1

    def close(self):
        if self.exchange is not None and hasattr(self.exchange, "close"):
            self.exchange.close()
        self.NN.close()


def timed_steps(job, lib, stream, flush, steps, warmup, world, sampler=None, phases_out=None):
    """W untimed + K timed steps, each bracketed by CUDA events on the launching stream, L2 flushed between
    iterations (outside the event pairs).  Returns (sum of step ms on this rank, launches, wall seconds)."""
    import torch
    import torch.distributed as dist
    from mpb200 import _lib
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    launches0 = 0
    t_wall0 = 0.0
    def read_phases():
        # per-kernel times of the step just enqueued (events recorded inside the calls).  Read AFTER the next
        # iteration's flush has been enqueued: the host then waits for this step's last validity kernel while the
        # GPU still has the exchange and the flush to run, instead of idling the GPU at every step boundary.
        phases_out["table"] += np.array([lib.mpb200_last_ms_of(_lib.OP_TABLE, k) for k in range(5)])
        phases_out["points"].append(lib.mpb200_last_ms_of(_lib.OP_POINTS, 1))
        phases_out["edges"].append(lib.mpb200_last_ms_of(_lib.OP_EDGES, 1))

    job.exchange_ms = []
    for it in range(warmup + steps):
        if it == warmup:
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            if sampler is not None:
                sampler.start()
            launches0 = lib.mpb200_launch_count()
            t_wall0 = time.perf_counter()
            job.exchange_ms = []
        flush.zero_()  # L2 flush between iterations (outside the event pair)
        if it > warmup and phases_out is not None:
            read_phases()
        if it >= warmup:
            ev[it - warmup][0].record(stream)
        job.step()
        if it >= warmup:
            ev[it - warmup][1].record(stream)
            if sampler is not None and sampler.nv and (it - warmup) % 8 == 0:
                sampler._sample()   # also from this thread, between steps (outside the event pairs): the region is short
    if phases_out is not None:
        read_phases()
        phases_out["exchange"] = list(job.exchange_ms[1:])   # the first entry belongs to the last warm-up step
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    launches = lib.mpb200_launch_count() - launches0
    return float(np.sum([a.elapsed_time(b) for a, b in ev])), int(launches), t_wall


def parity_check(job, rank, world, windows=4, width=256):
    """After the timed region: the table this rank just built (and, for N > 1, the GATHERED global colptr and
    validity bits) against the CPU oracle on sampled column windows.  Raises on any mismatch."""
    import torch
    from oracle import oracle as orc
    import fixtures as fx
    from mpb200 import sharding
    V, r, q0, q1 = job.V, job.r, job.q0, job.q1
    N = len(V)
    tree = orc.KDTree(V)
    O = orc.Obstacles2D(fx.ISRR_2H)
    So = orc.StateSpace([0, 0], [1, 1])
    colptr, rowval, nzval, words = sharding.table_device_tensors(job.NN.table)
    cp = colptr.cpu().numpy()
    bits = np.unpackbits(words.cpu().numpy().view(np.uint8), bitorder="little") if words is not None else np.zeros(0, np.uint8)
    checked = 0
    gcol = gbits = None
    if world > 1:
        gcol, gchunks = job.exchange.assemble()
        gbits = np.unpackbits(gchunks.view(np.uint8), bitorder="little")
        if len(gcol) != N + 1:
            raise RuntimeError("PARITY FAILURE: gathered colptr has %d entries for %d samples" % (len(gcol), N))
    ncols = q1 - q0
    starts = [int(x) for x in np.linspace(0, max(ncols - width, 0), windows)]
    for a in starts:
        b = min(a + width, ncols)
        ref_cp, ref_rv, ref_nz = tree.rball(r, q0 + a, q0 + b)
        lo, hi = int(cp[a]) - 1, int(cp[b]) - 1
        ok = np.array_equal(cp[a:b + 1] - cp[a], ref_cp - ref_cp[0])
        ok = ok and np.array_equal(rowval[lo:hi].cpu().numpy(), ref_rv)
        ok = ok and nzval[lo:hi].cpu().numpy().tobytes() == np.ascontiguousarray(ref_nz).tobytes()
        exp, _ = orc.edges_free_csc(O, So, V, ref_cp, ref_rv, q0 + a)
        ok = ok and np.array_equal(bits[lo:hi], np.asarray(exp, dtype=np.uint8))
        if not ok:
            raise RuntimeError("PARITY FAILURE (rank %d): shard columns [%d, %d) differ from the oracle" % (rank, q0 + a, q0 + b))
        checked += b - a
    if world > 1:
        # the gathered global structures, on windows inside EVERY rank's range (this is what proves the exchange)
        for g in range(world):
            g0, g1 = sharding.shard_range(N, g, world)
            for a in (g0, max(g1 - width, g0)):
                b = min(a + width, g1)
                ref_cp, ref_rv, _ = tree.rball(r, a, b)
                ok = np.array_equal(gcol[a:b + 1] - gcol[a], ref_cp - ref_cp[0])
                exp, _ = orc.edges_free_csc(O, So, V, ref_cp, ref_rv, a)
                lo, hi = int(gcol[a]) - 1, int(gcol[b]) - 1
                ok = ok and np.array_equal(gbits[lo:hi], np.asarray(exp, dtype=np.uint8))
                if not ok:
                    raise RuntimeError("PARITY FAILURE (rank %d): gathered columns [%d, %d) of rank %d differ from the oracle"
                                       % (rank, a, b, g))
                checked += b - a
    return checked


def dump_outputs(job, out_dir, sample_cols=32768):
    """What the last timed step left for its caller, as DIR/<name>.npy (float64; float32 for bits): this rank's
    colptr and point validity in full, and rowval / nzval / edge validity of the entries of a fixed, seeded sample
    of columns (the full table is ~28M entries per 1M columns).  Integers are exact in float64."""
    import torch
    from mpb200 import sharding
    os.makedirs(out_dir, exist_ok=True)
    colptr, rowval, nzval, words = sharding.table_device_tensors(job.NN.table)
    cp = colptr.cpu().numpy()
    ncols = len(cp) - 1
    cols = np.sort(np.random.Generator(np.random.PCG64(SEED)).choice(ncols, min(sample_cols, ncols), replace=False))
    # 0-based positions of every entry of the sampled columns
    idx = np.concatenate([np.arange(cp[j] - 1, cp[j + 1] - 1) for j in cols])
    ti = torch.from_numpy(idx).to(colptr.device)
    e_bits = (words[ti >> 6] >> (ti & 63)) & 1
    # the step enqueues K6 with its bits left on the device; fetching them re-runs the same pure per-sample test
    p_bits = np.unpackbits(job.NN.points_free(job.CC, job.SS).view(np.uint8), bitorder="little")[:ncols]
    arrays = {"colptr": cp.astype(np.float64), "point_free": p_bits.astype(np.float32),
              "sample_columns": cols.astype(np.float64),
              "sample_rowval": rowval[ti].cpu().numpy().astype(np.float64),
              "sample_nzval": nzval[ti].cpu().numpy(),
              "sample_edge_free": e_bits.cpu().numpy().astype(np.float32)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def allreduce_max_sum(vals_max, vals_sum, world):
    import torch
    import torch.distributed as dist
    tm = torch.tensor(vals_max, dtype=torch.float64, device="cuda")
    ts = torch.tensor(vals_sum, dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(ts, op=dist.ReduceOp.SUM)
    return [float(x) for x in tm], [float(x) for x in ts]


def mc_leg(mp, lib, rank, world, n_total=100_000_000):
    """configs[4]: 1e8 importance-sampled rollouts sharded by rollout id (Philox keyed by the global id: the
    shard layout does not change any draw), sums all-reduced.  Device-timed: the rollout kernel's own CUDA events
    (max over ranks) + the all-reduce between events."""
    import torch
    import torch.distributed as dist
    import bench_configs as bc
    from mpb200 import _lib, sharding
    P, CC, _ = bc.c5_problem(mp)
    a, b = sharding.shard_range(n_total, rank, world)
    mp.collision_probability(P, CC, 200_000, first=a)       # warm-up
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    res = mp.collision_probability(P, CC, b - a, first=a)
    k_ms = lib.mpb200_last_ms_of(_lib.OP_OTHER, 0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    tot = sharding.allreduce_mc(res) if world > 1 else dict(res)
    e1.record()
    torch.cuda.synchronize()
    (k_max, r_max), _ = allreduce_max_sum([k_ms, e0.elapsed_time(e1)], [0.0], world)
    ms = k_max + (r_max if world > 1 else 0.0)
    n = max(int(tot["n"]), 1)
    p = tot["S1"] / n
    return {"config": "C5 / configs[4]: Monte-Carlo collision probability, T=%d, K=%d, %d rollouts sharded by rollout id x%d + all-reduce of (S1, S2, S0, n, hits)"
                      % (P.T, P.K, n_total, world),
            "metric": "rollouts_per_sec", "value": n_total / (ms / 1e3), "unit": "rollouts/s", "ms": ms,
            "kernel_ms_max_over_ranks": k_max, "allreduce_ms": r_max if world > 1 else 0.0,
            "rollouts": int(tot["n"]), "hits": int(tot["hits"]), "p": p,
            "se": (max(tot["S2"] / n - p * p, 0.0) / n) ** 0.5, "S1": tot["S1"],
            "note": "hits is an integer count and must be identical for every GPU count; S1/S2 agree to summation order"}


# ---------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the C3/C4/C5 secondary block (N = 1) and the MC leg")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="headline line: weak (N x 1M samples) or strong (1M samples in total); the other one is still reported as a sub-object")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0's columns) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import mpb200
    from mpb200 import _lib, sharding

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = mpb200.init(local)
    # ONE explicit stream for everything in the timed region: the L2 flush, the timing events, the library's
    # kernels and (N > 1) the exchange.  (torch's default stream has handle 0, which mpb200_set_stream
    # reads as "use the library's own non-blocking stream": the flush would then overlap the step.)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    _lib.check(lib.mpb200_set_stream(_lib.c_vp(stream.cuda_stream)))
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def build_job(n_total, tag):
        samples = make_samples(n_total, world > 1)
        V = torch.from_numpy(samples).pin_memory().numpy()
        q0, q1 = sharding.shard_range(n_total, rank, world)
        return Job(mpb200, V, q0, q1, world, tag)

    # ---- the two multi-GPU readings of C2: weak (headline by default) and strong (configs[1] literally)
    n_weak, n_strong = SAMPLES_PER_GPU * world, SAMPLES_PER_GPU
    head_n = n_weak if args.scaling == "weak" else n_strong
    job = build_job(head_n, "head")
    phases = {"table": np.zeros(5), "points": [], "edges": [], "exchange": []}
    sampler = ClockSampler(local)
    total_ms, launches, t_wall = timed_steps(job, lib, stream, flush, args.steps, args.warmup, world, sampler, phases)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(job, args.dump_outputs)
    nnz = job.nnz
    (total_ms_max,), (edges_all,) = allreduce_max_sum([total_ms], [float(nnz)], world)
    per_rank = None
    if world > 1:   # every rank's own view of the step (its event total and kernel phases): shows skew and who waits
        mine = torch.tensor([total_ms / args.steps, phases["table"][0] / args.steps, float(np.mean(phases["points"])),
                             float(np.mean(phases["edges"])),
                             float(np.mean(phases["exchange"])) if phases["exchange"] else 0.0, float(nnz)],
                            dtype=torch.float64, device="cuda")
        allr = torch.empty(world * mine.numel(), dtype=torch.float64, device="cuda")
        dist.all_gather_into_tensor(allr, mine)
        per_rank = [dict(zip(("ms_per_step", "inball_total", "points", "edges", "exchange_incl_wait", "edges_built"), row))
                    for row in allr.cpu().numpy().reshape(world, -1).round(4).tolist()]
    ms_per_step = total_ms_max / args.steps
    value = edges_all / (ms_per_step / 1e3)
    parity_cols = parity_check(job, rank, world)
    (_,), (parity_all,) = allreduce_max_sum([0.0], [float(parity_cols)], world)

    # what the output format alone costs: the table's write pattern without any neighbour work (csrc/peaks.cu)
    write_floor_ms = None
    if rank == 0:
        import ctypes
        v = ctypes.c_double(0.0)
        if lib.mpb200_table_write_floor(job.NN.table.h, ctypes.byref(v)) == 0:
            write_floor_ms = v.value

    other = None
    if world > 1:
        # the other scaling mode, same code path, fewer steps
        o_n = n_strong if args.scaling == "weak" else n_weak
        ojob = build_job(o_n, "other")
        o_steps = max(10, args.steps // 2)
        o_ms, _, _ = timed_steps(ojob, lib, stream, flush, o_steps, 3, world)
        (o_max,), (o_edges,) = allreduce_max_sum([o_ms], [float(ojob.nnz)], world)
        o_par = parity_check(ojob, rank, world, windows=2)
        (_,), (o_par_all,) = allreduce_max_sum([0.0], [float(o_par)], world)
        other = {"scaling": "strong" if args.scaling == "weak" else "weak", "n_samples_total": o_n,
                 "query_columns_per_gpu": o_n // world, "steps": o_steps, "ms_per_step": o_max / o_steps,
                 "value": o_edges / (o_max / o_steps / 1e3), "unit": UNIT,
                 "nn_queries_per_sec": o_n / (o_max / o_steps / 1e3), "edges_per_step": o_edges,
                 "exchange": ojob.exchange_kind, "parity_checked": int(o_par_all)}
        ojob.close()

    mc = None
    if not args.no_secondary:
        mc = mc_leg(mpb200, lib, rank, world)

    # ---- auxiliary figure: the SAME samples numbered along a Z-order curve (what mpb200_sample_free's Morton
    # option produces).  FMT* does not care how i.i.d. samples are numbered; the kernels do (column writes and
    # gathers become local).  Reported beside the headline, never instead of it.
    renumbered = None
    if world == 1:
        V = job.V
        NNm = mpb200.MetricNN(np.ascontiguousarray(V[morton_order(V)]))
        NNm.handle()
        evm = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
        for it in range(3 + len(evm)):
            flush.zero_()
            if it >= 3:
                evm[it - 3][0].record(stream)
            NNm.points_free(job.CC, job.SS, fetch=False)
            nnz_m = NNm.build_table(job.r)
            NNm.edges_free(NNm.table, job.CC, job.SS, fetch=False, count=False)
            if it >= 3:
                evm[it - 3][1].record(stream)
        torch.cuda.synchronize()
        ms_m = float(np.mean([a.elapsed_time(b) for a, b in evm]))
        renumbered = {"order": "Z-order (Morton) numbering of the same samples", "ms_per_step": ms_m,
                      "value": nnz_m / (ms_m / 1e3), "unit": UNIT, "steps": len(evm)}
        NNm.close()

    # ---- end to end through the public API with HOST buffers (H2D + D2H inside the timed region)
    e2e_times = []
    V = job.V
    h2d = V.nbytes
    d2h = 0
    pool = _lib.PinnedPool(reuse=True)    # the benchmark loop's explicit opt-in: result buffers reused across steps
    for it in range(2 + args.e2e_steps):
        NN2 = mpb200.MetricNN(V)          # fresh sample set: H2D of the inputs is inside
        NN2.pool = pool
        NN2.set_query_range(job.q0, job.q1)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        cache, Eb, _ = NN2.precompute_checked(job.r, job.CC, job.SS)   # H2D samples, fused build, D2H colptr/rowval/nzval/edge bits
        Fb = NN2.points_free(job.CC, job.SS)      # D2H point bits
        t1 = time.perf_counter()
        if it >= 2:
            e2e_times.append(t1 - t0)
        d2h = cache.D.colptr.nbytes + cache.D.rowval.nbytes + cache.D.nzval.nbytes + Fb.nbytes + Eb.nbytes
        NN2.pool = _lib.PinnedPool()
        NN2.close()
    (e2e_s,), _ = allreduce_max_sum([float(np.mean(e2e_times))], [0.0], world)
    e2e_value = edges_all / e2e_s

    if rank == 0:
        peak, peak_kind = peaks()
        ncols = job.q1 - job.q0
        deg = nnz / ncols
        fill_ms = phases["table"][4] / args.steps
        alg_bytes = (8 * 2 + 8 + 16 * deg) * ncols   # SURVEY 8(d): 8d + 8 + 16*deg per query
        achieved = alg_bytes / (fill_ms / 1e3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(head_n, job.r),
                       "l2": "512 MiB flush between timed iterations", "index_type": "int64 (reference ABI)",
                       "parallelism": "query-range shards x%d (samples in stripe order when x > 1), samples+obstacles replicated%s"
                                      % (world, ", per step: column lengths + validity words of every rank to every rank (%s)"
                                         % job.exchange_kind if world > 1 else "")},
            "nn_queries_per_sec": head_n / (ms_per_step / 1e3),
            "edges_per_step": edges_all, "mean_degree": deg,
            "phase_ms": {"grid_build": phases["table"][1] / args.steps, "count_scan": phases["table"][2] / args.steps,
                         "host_gap": phases["table"][3] / args.steps, "fill": fill_ms,
                         "points_kernel": float(np.mean(phases["points"])), "edges_kernels": float(np.mean(phases["edges"])),
                         "inball_total": phases["table"][0] / args.steps,
                         "exchange": float(np.mean(phases["exchange"])) if phases["exchange"] else None},
            "exchange": job.exchange_kind,
            "per_rank": per_rank,
            "parity_checked": int(parity_all),
            "gpu_launches": launches,
            "renumbered_samples": renumbered,
            "strong_scaling" if args.scaling == "weak" else "weak_scaling": other,
            "mc": mc,
            "wall_ms_per_step_incl_flush": 1e3 * t_wall / args.steps,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": 1e3 * e2e_s, "steps": args.e2e_steps,
                    "note": "d2h_bytes_per_step = bytes delivered into the caller's Int64 / Float64 / BitVector arrays (the "
                            "reference's formats); the Int64 row indices cross PCIe bit-packed (20 bits each at N = 1M) and "
                            "are unpacked into the caller's array by host threads during the nzval transfer"},
            "roofline": {"kernel": "rball_fill<2>", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": fill_traffic(), "peak_kind": peak_kind,
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "write_pattern_floor_ms": write_floor_ms, "kernel_ms": fill_ms,
                         "frac_of_write_pattern_floor": (write_floor_ms / fill_ms) if write_floor_ms else None,
                         "note": "write_pattern_floor = a kernel that only writes the same column bursts in the same order "
                                 "(mpb200_table_write_floor): the cost of the reference's CSC format for samples numbered as drawn"},
        }
        if world == 1 and not args.no_cpu_baseline:
            # the oracle port on this box's host cores: full workload, single thread (the reference is
            # single-threaded) -- reported baseline only
            e1, tb1, tq1 = run_oracle(V, job.r, 0, SAMPLES_PER_GPU, 1)
            line["cpu_baseline"] = {"value": e1 / (tb1 + tq1), "unit": UNIT, "cores": 1, "kind": "port",
                                    "sample": "full workload: kd-tree build %.2fs + %d query columns, %d edges in %.2fs"
                                              % (tb1, SAMPLES_PER_GPU, e1, tq1),
                                    "host_cores_available": host_threads()}
    job.close()
    if rank == 0:
        if world == 1 and not args.no_secondary:
            line["secondary"] = secondary_block(mpb200, lib)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def secondary_block(mp, lib):
    """BASELINE.json configs C3 / C4 / C5 at full size on this GPU: device-resident time, own roofline, own
    cpu_baseline (oracle port, bounded sample), parity against the oracle on the sample.  Each entry is
    self-describing; a failure of one config is reported, not hidden."""
    import types
    import bench_configs as bc
    from oracle import oracle as orc
    import fixtures as fx
    from mpb200 import _lib
    _lib.check(lib.mpb200_release_cached())
    out = {}
    args = types.SimpleNamespace(scale=1.0)
    for name, fn in (("C3", bc.c3), ("C4", bc.c4), ("C5", bc.c5), ("F4", bc.f4), ("KNN", bc.kn)):
        try:
            out[name] = fn(mp, orc, fx, args)
        except Exception as e:   # noqa: BLE001 -- report and go on: the headline line must still print
            out[name] = {"config": name, "error": "%s: %s" % (type(e).__name__, e)}
        _lib.check(lib.mpb200_release_cached())
    out["peaks"] = {"fp64_dadd_dmul_gops": bc.pipe_peak(lib, 0) / 1e9, "fp64_dfma_gflops": bc.pipe_peak(lib, 1) / 1e9,
                    "fp32_ffma_gflops": bc.pipe_peak(lib, 2) / 1e9,
                    "how": "mpb200_pipe_peak: register-resident dependency-free streams on every SM, CUDA-event timed (csrc/peaks.cu)"}
    return out


if __name__ == "__main__":
    main()
