#!/usr/bin/env python
"""Roadmap-optimal plans (PRM*, mpb200_sssp_plan) against GMT* in table mode (mpb200_gmt_plan) over the same device
roadmap, on three workloads:
  C2    2-D unit square, ISRR_2H, N = 1M free samples (sample_free, seed 20240602), BallGoal((.9, .9), .01), r = fmt_radius
  RS    Reeds-Shepp, N = 200k SE2 states (seed 20240605), ISRR_2H, turning radius 0.01, r = 0.025
  C4    double integrator (4-D state), N = 200k states (seed 20240604), ISRR_2H, r = 0.734
(the workloads of scripts/gmt_lazy_bench.py).  The roadmap is built once by planners.prmstar; then the PRM* plan and the
GMT* plan at lambda = 1 are called alternately on its tables, --reps times after one warm-up of each, and the medians
of their device times (CUDA events, MPB200_OP_PLAN) are recorded with rounds, levels, |R| and, for lambda in
{0.5, 1, 2}, GMT* cost over PRM* cost.  Every repetition's outputs are asserted equal.  The GPU's name and power limit
are read in the same run.  Prints one JSON line; --out writes it to a file too.

  python scripts/sssp_bench.py [--reps 5] [--out profiles/sssp/bench.json]
"""
import argparse
import ctypes
import json
import os
import statistics
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import mpb200 as mp  # noqa: E402
from mpb200 import _lib  # noqa: E402
from gmt_lazy_bench import c2, c4, cars, gpu_info  # noqa: E402


def calls(P):
    """-> (prm(), gmt(lam)) over the tables prmstar left on the device, each returning (outputs, device ms)"""
    NN = P.V
    DF, DB = (NN.tableF, NN.tableB) if hasattr(NN, "tableF") else (NN.table, NN.table)
    N = len(NN)
    from mpb200.planners import _goal_chunks
    chunks = _goal_chunks(NN.V, P.goal, P.SS)
    r = P.solution.metadata["r"]
    lib = _lib.lib()
    path, tree, C = np.empty(N, np.int64), np.empty(N, np.int64), np.empty(N)

    def prm():
        desc = _lib.GmtDesc(DF.h, DB.h, _lib.ptr(chunks), 1, 0.0, 1, None)
        res = _lib.SsspResult()
        _lib.check(lib.mpb200_sssp_plan(NN.handle(), ctypes.byref(desc), ctypes.byref(res), _lib.ptr(path), N,
                                        _lib.ptr(tree), _lib.ptr(C)))
        out = (res.solved, res.cost, res.rounds, res.levels, res.reached, res.grid_blocks,
               path[:res.path_len].tobytes(), tree.tobytes(), C.tobytes())
        return out, lib.mpb200_last_ms_of(_lib.OP_PLAN, 0)

    def gmt(lam):
        desc = _lib.GmtDesc(DF.h, DB.h, _lib.ptr(chunks), 1, lam * r, 1, None)
        res = _lib.GmtResult()
        _lib.check(lib.mpb200_gmt_plan(NN.handle(), ctypes.byref(desc), ctypes.byref(res), _lib.ptr(path), N,
                                       _lib.ptr(tree), _lib.ptr(C)))
        out = (res.solved, res.cost, res.iterations, path[:res.path_len].tobytes(), tree.tobytes(), C.tobytes())
        return out, lib.mpb200_last_ms_of(_lib.OP_PLAN, 0)

    return prm, gmt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--n1", type=int, default=1_000_000)
    ap.add_argument("--n2", type=int, default=200_000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    mp.init(0)
    line = dict(gpu=gpu_info(), note="device ms = CUDA events around the one cooperative launch of each plan "
                                     "(MPB200_OP_PLAN); PRM* and GMT* (table mode, lambda = 1) alternated over the "
                                     "same roadmap, medians of %d after one warm-up of each" % a.reps)
    work = {
        "C2": ("2-D unit square, ISRR_2H, N=%d, BallGoal((.9,.9),.01), r=fmt_radius" % a.n1, c2(a.n1)),
        "RS": ("Reeds-Shepp, N=%d SE2 states, ISRR_2H, turning radius 0.01, r=0.025" % a.n2, cars("reedsshepp", a.n2)),
        "C4": ("double integrator (4-D state), N=%d, ISRR_2H, r=0.734" % a.n2, c4(a.n2)),
    }
    for name, (desc, (make, kw)) in work.items():
        P = make()
        st, cost, elapsed = mp.prmstar(P, **kw)
        m = P.solution.metadata
        prm, gmt = calls(P)
        p0, _ = prm()
        g0, _ = gmt(1.0)
        pms, gms = [], []
        for _ in range(a.reps):
            o, t = prm()
            assert o == p0
            pms.append(t)
            o, t = gmt(1.0)
            assert o == g0
            gms.append(t)
        ratios = {}
        for lam in (0.5, 1.0, 2.0):
            g, _ = gmt(lam)
            ratios[str(lam)] = (g[1] / p0[1]) if (g[0] and p0[0]) else None
            assert not g[0] or g[1] >= p0[1]
        line[name] = dict(
            workload=desc, status=st, cost=cost, from_scratch_s=elapsed, r=m["r"], grid_blocks=p0[5],
            prm_plan_ms=statistics.median(pms), prm_plan_ms_all=pms, gmt_plan_ms=statistics.median(gms),
            gmt_plan_ms_all=gms, gmt_iterations=g0[2], rounds=p0[2], levels=p0[3], reached=p0[4],
            path_len=len(m["path"]), gmt_cost_over_prm_cost=ratios)
        P.V.close()
    line["gpu_after"] = gpu_info()
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
