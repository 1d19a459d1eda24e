#!/usr/bin/env python
"""GMT* on the device (mpb200_gmt_plan) at config C2: 2-D unit square, ISRR_2H, N = 1M samples, r from fmt_radius.

Prints one JSON line:
  per lambda in {0.5, 1, 2}: the plan's device time (CUDA events around the planning kernel, after one warm-up plan,
  median of --reps re-plans over the resident tables), iterations, expansions, checks, the from-scratch time
  (host clock around gmtstar on a fresh problem: sample_free + checked table build + point bits + plan + path + the
  tree and costs, ending in a synchronise) and the GMT*/FMT* cost ratio on the same samples;
  host fmtstar(edge_checks="table") wall time at N = 100k and, run once, at N = 1M;
  the GPU's name and power limit.

  python scripts/gmt_bench.py [--reps 10] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mpb200 as mp  # noqa: E402
from mpb200 import _lib  # noqa: E402
from mpb200.problems import goal_mask  # noqa: E402

SEED = 20240602
LAMBDAS = (0.5, 1.0, 2.0)


def problem(V=None):
    SS = mp.UnitHypercube(2)
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    kw = {} if V is None else dict(V=mp.MetricNN(V, SS.dist, V[0]))
    return mp.MPProblem(SS, [0.1, 0.1], mp.BallGoal([0.9, 0.9], 0.01), CC, **kw)


def replan_ms(P, lam, reps):
    """device time of the planning kernel over the tables gmtstar left resident, median of reps"""
    NN, N = P.V, len(P.V)
    chunks = np.zeros((N + 63) // 64 * 8, dtype=np.uint8)
    pk = np.packbits(goal_mask(NN.V, P.goal, P.SS), bitorder="little")
    chunks[:len(pk)] = pk
    chunks = chunks.view(np.uint64)
    space = P.SS.desc()
    desc = _lib.GmtDesc(NN.table.h, NN.table.h, _lib.ptr(chunks), 1, lam * P.solution.metadata["r"], 1,
                        ctypes.pointer(space))
    res = _lib.GmtResult()
    path = np.empty(N, dtype=np.int64)
    lib = _lib.lib()
    ms = []
    for _ in range(reps + 1):
        _lib.check(lib.mpb200_gmt_plan(NN.handle(), ctypes.byref(desc), ctypes.byref(res), _lib.ptr(path), N,
                                       None, None))
        ms.append(lib.mpb200_last_ms_of(_lib.OP_PLAN, 1))
    return statistics.median(ms[1:]), res


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--N", type=int, default=1_000_000)
    ap.add_argument("--fmt-small", type=int, default=100_000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    mp.init(0)
    N = a.N
    # warm-up: modules, block cache, the first cooperative launch
    P0 = problem()
    mp.gmtstar(P0, 20_000, lam=1.0, seed=SEED)
    P0.V.close()

    runs = {}
    V = None
    for lam in LAMBDAS:
        P = problem()
        st, cost, elapsed = mp.gmtstar(P, N, lam=lam, seed=SEED)       # from scratch, ends in a synchronise
        m = P.solution.metadata
        dev_ms, res = replan_ms(P, lam, a.reps)
        assert res.iterations == m["iterations"] and res.cost == cost
        runs[str(lam)] = dict(status=st, cost=cost, from_scratch_s=elapsed, plan_device_ms=dev_ms,
                              iterations=m["iterations"], expansions=m["expansions"], checks=m["checks"],
                              path_len=len(m["path"]), r=m["r"], grid_blocks=m["grid_blocks"])
        if V is None:
            V = P.V.V.copy()
        P.V.close()

    Pf = problem(V)                                                   # FMT* on the same 1M samples, once
    t0 = time.perf_counter()
    st_f, cost_f, _ = mp.fmtstar(Pf, edge_checks="table")
    fmt_1m_s = time.perf_counter() - t0
    Pf.V.close()
    for lam in LAMBDAS:
        runs[str(lam)]["cost_ratio_vs_fmtstar"] = runs[str(lam)]["cost"] / cost_f

    Ps = problem()
    t0 = time.perf_counter()
    mp.fmtstar(Ps, a.fmt_small, seed=SEED, edge_checks="table")
    fmt_small_s = time.perf_counter() - t0
    Ps.V.close()

    line = dict(workload="C2: GMT* 2-D unit square, ISRR_2H, N=%d, BallGoal((.9,.9), .01), r=fmt_radius" % N,
                gpu=gpu_info(), lambdas=runs, fmtstar_cost=cost_f, fmtstar_status=st_f,
                fmtstar_host_wall_s={"%d" % a.fmt_small: fmt_small_s, "%d" % N: fmt_1m_s},
                plan_device_ms_note="CUDA events around the planning kernel, median of %d re-plans after one" % a.reps)
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
