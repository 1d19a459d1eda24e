#!/usr/bin/env python
"""Shortcutting planned C2 paths on the device (mpb200_shortcut_paths).

  workload  C2 (2-D unit square, ISRR_2H, N = 1M free samples, seed 20240602, r = fmt_radius), lambda = 1: the 64 random
            queries of scripts/gmt_batch_bench.py (seed 7: random free inits, BallGoal(radius 0.01) at random free
            samples) through gmtstar_batch, then one batched call on the solved paths for k in {1, 4, 8}.
  records   per k: device ms of the call and of each phase (CUDA events; medians of --reps after one warm-up), pairs and
            segment tests, min / mean / max of output cost over planned cost, the same paths shortcut one call each
            (sum of their device times) against the batched call (outputs asserted equal), and the time the CPU
            restatement of the tests (tests/oracle_shortcut.py) takes on a few paths -- test infrastructure, not a
            baseline.  The GPU's name and power limit are read in the same run.
Prints one JSON line; --out writes it to a file too.

  python scripts/shortcut_bench.py [--reps 5] [--out profiles/shortcut/bench.json]
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
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def call(lib, _lib, CC, SS, paths, k):
    """one mpb200_shortcut_paths call -> (outputs, device ms of the call, phase 1, phase 2)"""
    n, d = len(paths), SS.dim
    offs = np.zeros(n + 1, dtype=np.int64)
    offs[1:] = np.cumsum([len(p) for p in paths])
    Y = np.ascontiguousarray(np.vstack(paths))
    cap = max((len(p) - 1) * k + 1 for p in paths)
    out = np.empty((n, cap, d))
    ol, co, pa, sc = np.empty(n, np.int64), np.empty(n), np.empty(n, np.int64), np.empty(n, np.int64)
    space = SS.desc()
    _lib.check(lib.mpb200_shortcut_paths(_lib.ptr(Y), _lib.ptr(offs), n, d, CC.handle(), ctypes.byref(space), k,
                                         _lib.ptr(out), cap, _lib.ptr(ol), _lib.ptr(co), _lib.ptr(pa), _lib.ptr(sc)))
    ms = [lib.mpb200_last_ms_of(_lib.OP_PATH, p) for p in range(3)]
    outs = [(int(ol[q]), out[q, :ol[q]].tobytes(), float(co[q]), int(pa[q]), int(sc[q])) for q in range(n)]
    return outs, ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--oracle-paths", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import mpb200 as mp
    from mpb200 import _lib
    lib = mp.init(0)
    line = dict(gpu=gpu_info(), note="device ms = CUDA events around the call's kernels (phase 1: nodes + visibility, "
                                     "phase 2: minimum + output rows); medians of %d runs after a warm-up" % a.reps)
    N = 1_000_000
    SS = mp.UnitHypercube(2)
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    P = mp.MPProblem(SS, [0.1, 0.1], mp.BallGoal([0.9, 0.9], 0.01), CC)
    mp.gmtstar(P, N, lam=1.0, seed=20240602)                     # the roadmap, to pick free samples from (as the batch bench)
    V = P.V.V
    F = np.unpackbits(P.V.points_free(CC, SS).view(np.uint8), bitorder="little")[:N].astype(bool)
    free = np.flatnonzero(F)
    rng = np.random.Generator(np.random.PCG64(7))
    inits = rng.choice(free, 64) + 1
    centres = [V[j, :2].copy() for j in rng.choice(free, 64)]
    r = P.solution.metadata["r"]                                 # the same roadmap: same samples, same radius
    sols = mp.gmtstar_batch(P, [int(i) for i in inits], [mp.BallGoal(c, 0.01) for c in centres], lam=1.0, r=r,
                            trees=False)
    assert np.array_equal(P.V.V, V) and all(s.metadata.get("r", r) == r for s in sols)
    solved = [s for s in sols if s.status == "solved"]
    paths = [np.ascontiguousarray(V[np.asarray(s.metadata["path"]) - 1]) for s in solved]
    planned = np.array([s.cost for s in solved])
    lens = [len(p) for p in paths]
    line["paths"] = dict(queries=64, solved=len(solved), vertices_min=min(lens), vertices_mean=float(np.mean(lens)),
                         vertices_max=max(lens), r=solved[0].metadata["r"])
    line["k"] = {}
    for k in (1, 4, 8):
        call(lib, _lib, CC, SS, paths, k)                           # warm-up
        runs = [call(lib, _lib, CC, SS, paths, k) for _ in range(a.reps)]
        outs = runs[-1][0]
        assert all(r[0] == outs for r in runs)
        singles_ms = []
        for _ in range(a.reps):
            tot = 0.0
            for q, p in enumerate(paths):
                o, ms = call(lib, _lib, CC, SS, [p], k)
                assert o[0] == outs[q], "a path alone differs from the batched call"
                tot += ms[0]
            singles_ms.append(tot)
        ratio = np.array([o[2] for o in outs]) / planned
        assert np.all(ratio <= 1.0)
        med = lambda i: statistics.median(r[1][i] for r in runs)
        line["k"][str(k)] = dict(
            call_ms=med(0), phase1_visibility_ms=med(1), phase2_minimum_ms=med(2),
            call_ms_all=[r[1][0] for r in runs], singles_sum_ms=statistics.median(singles_ms),
            singles_sum_ms_all=singles_ms, batched_vs_singles=statistics.median(singles_ms) / med(0),
            pairs=int(sum(o[3] for o in outs)), segment_checks=int(sum(o[4] for o in outs)),
            nodes_max=max((n - 1) * k + 1 for n in lens),
            cost_ratio_min=float(ratio.min()), cost_ratio_mean=float(ratio.mean()), cost_ratio_max=float(ratio.max()),
            output_vertices_mean=float(np.mean([o[0] for o in outs])))
    # the CPU restatement on a few paths (test infrastructure, not a baseline)
    from oracle import oracle as orc
    import fixtures as fx
    from oracle_shortcut import shortcut_oracle
    O, So = orc.Obstacles2D(fx.ISRR_2H), orc.StateSpace([0, 0], [1, 1])
    t0 = time.perf_counter()
    for p in paths[:a.oracle_paths]:
        shortcut_oracle(orc, O, So, p, 4)
    line["cpu_restatement_k4"] = dict(paths=a.oracle_paths, seconds=time.perf_counter() - t0,
                                      note="tests/oracle_shortcut.py (test infrastructure, not a baseline)")
    line["gpu_after"] = gpu_info()
    P.V.close()
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
