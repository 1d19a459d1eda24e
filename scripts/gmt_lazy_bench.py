#!/usr/bin/env python
"""Lazy against table GMT* (planners.gmtstar(edge_checks="lazy" | "table")) on four workloads, lambda = 1:
  C2    2-D unit square, ISRR_2H, N = 1M free samples (sample_free, seed 20240602), BallGoal((.9, .9), .01), r = fmt_radius
  RS    Reeds-Shepp, N = 200k SE2 states (the F4 set of bench_configs.py + init and goal), turning radius 0.01, r = 0.025
  DUB   Dubins, the same states and radii
  C4    double integrator (4-D state), N = 200k states (the C4 set of bench_configs.py + init and goal), r = 0.734
each past ISRR_2H.  Per workload and mode, alternating the modes, after one warm-up plan of each: the median time from
scratch (host clock around gmtstar on a fresh problem: tables, edge pass in table mode, point bits, plan, tree and
costs, ending in a synchronise), the median device time of the plan (CUDA events around the planning kernel), and the
segment tests: table mode runs the edge pass over every stored edge of the backward table, lazy mode only those of the
motions it uses.  Asserts that both modes return the same tree, costs and path bytes.  Reads the GPU's name and power
limit in the same run and prints one JSON line.

  python scripts/gmt_lazy_bench.py [--reps 5] [--out profiles/gmt/lazy_bench.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mpb200 as mp  # noqa: E402


def c2(N):
    SS = mp.UnitHypercube(2)
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    return lambda: mp.MPProblem(SS, [0.1, 0.1], mp.BallGoal([0.9, 0.9], 0.01), CC), dict(N=N, seed=20240602)


def cars(kind, N):
    rng = np.random.Generator(np.random.PCG64(20240605))
    V = np.column_stack([rng.random(N - 2), rng.random(N - 2), rng.uniform(0, 2 * np.pi, N - 2)])
    V = np.vstack([[0.1, 0.1, 0.0], V, [0.9, 0.9, 0.0]])
    SS = (mp.ReedsSheppMetricSpace if kind == "reedsshepp" else mp.DubinsQuasiMetricSpace)(0.01)
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    NNcls = mp.MetricNN if kind == "reedsshepp" else mp.QuasiMetricNN
    return lambda: mp.MPProblem(SS, V[0], mp.StateGoal(V[-1]), CC, V=NNcls(V, SS.dist, V[0])), dict(r=0.025)


def c4(N):
    rng = np.random.Generator(np.random.PCG64(20240604))
    SS = mp.DoubleIntegrator(2)
    V = SS.lo + rng.random((N - 2, 4)) * (SS.hi - SS.lo)
    V = np.vstack([[0.1, 0.1, 0.0, 0.0], V, [0.9, 0.9, 0.0, 0.0]])
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    return lambda: mp.MPProblem(SS, V[0], mp.StateGoal(V[-1]), CC, V=mp.QuasiMetricNN(V, SS.dist, V[0])), dict(r=0.734)


def plan(make, kw, mode):
    P = make()
    st, cost, elapsed = mp.gmtstar(P, lam=1.0, edge_checks=mode, **kw)
    m = P.solution.metadata
    out = dict(status=st, cost=cost, from_scratch_s=elapsed, plan_device_ms=m["device_ms"], iterations=m["iterations"],
               checks=m["checks"], collision_checks=m["collision_checks"], grid_blocks=m["grid_blocks"],
               segment_checks=m["segment_checks"] if mode == "lazy" else m["precomputed_edge_checks"])
    key = (m["tree"].tobytes(), m["costs"].tobytes(), np.asarray(m["path"], dtype=np.int64).tobytes())
    P.V.close()
    return out, key


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    mp.init(0)
    n1, n2 = int(1_000_000 * a.scale), int(200_000 * a.scale)
    workloads = {
        "C2": ("2-D unit square, ISRR_2H, N=%d, BallGoal((.9,.9),.01), r=fmt_radius" % n1, c2(n1)),
        "RS": ("Reeds-Shepp, N=%d SE2 states, ISRR_2H, turning radius 0.01, r=0.025" % n2, cars("reedsshepp", n2)),
        "DUB": ("Dubins, N=%d SE2 states, ISRR_2H, turning radius 0.01, r=0.025" % n2, cars("dubins", n2)),
        "C4": ("double integrator (4-D state), N=%d, ISRR_2H, r=0.734" % n2, c4(n2)),
    }
    result = {}
    for name, (desc, (make, kw)) in workloads.items():
        keys = {}
        for mode in ("table", "lazy"):                              # warm-up: modules, block cache, first launch
            _, keys[mode] = plan(make, kw, mode)
        runs = {"table": [], "lazy": []}
        for _ in range(a.reps):
            for mode in ("table", "lazy"):
                o, k = plan(make, kw, mode)
                assert k == keys[mode] == keys["table"], (name, mode)
                runs[mode].append(o)
        entry = dict(workload=desc, lam=1.0)
        for mode, rs in runs.items():
            entry[mode] = dict(rs[0], from_scratch_s=statistics.median(r["from_scratch_s"] for r in rs),
                               plan_device_ms=statistics.median(r["plan_device_ms"] for r in rs),
                               from_scratch_s_all=[r["from_scratch_s"] for r in rs],
                               plan_device_ms_all=[r["plan_device_ms"] for r in rs])
        entry["lazy_over_table_from_scratch"] = entry["lazy"]["from_scratch_s"] / entry["table"]["from_scratch_s"]
        entry["identical_tree_costs_path"] = True
        result[name] = entry
    line = dict(gpu=gpu_info(), reps=a.reps, workloads=result,
                note="segment_checks: table = the edge pass over every stored edge of the backward table; lazy = the "
                     "motions the plan uses.  Medians over reps, modes alternated in one process.")
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
