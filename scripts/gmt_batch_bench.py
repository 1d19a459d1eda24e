#!/usr/bin/env python
"""A batch of GMT* queries over one roadmap (mpb200_gmt_plan_batch) against the same queries planned one by one.

  scaling   C2 (2-D unit square, ISRR_2H, N = 1M free samples, seed 20240602, r = fmt_radius), lambda = 1, table and
            lazy mode, Q in {1, 4, 16, 64}: random free inits, BallGoal(radius 0.01) at random free samples.  Per Q,
            alternating the two, --reps times: the device time of the batch (CUDA events around its one planning
            kernel) and the sum of the device times of the Q single plans (mpb200_gmt_plan / _lazy); medians.  The
            iterations of the queries (max, mean) and an assertion that every query's outputs equal its single plan.
  cars      the same on Reeds-Shepp, N = 200k SE2 states, turning radius 0.01, r = 0.025, lazy mode (the edge test of
            each candidate is a car path checked by one lane).
  q1        the single-plan workloads of scripts/gmt_bench.py (C2 table, lambda 0.5 / 1 / 2) and
            scripts/gmt_lazy_bench.py (C2, RS, DUB, C4 lazy, lambda 1): median device time of --reps re-plans over
            resident tables, in child processes that alternate this tree with --parent-root (a built checkout of the
            parent commit), --rounds times each.
  api       gmtstar_batch(trees=False) from scratch with the 64 C2 queries, per mode: equal to the batch, wall time.
The GPU's name and power limit are read in the same run.  Prints one JSON line; --out writes it to a file too.

  python scripts/gmt_batch_bench.py [--reps 5] [--parent-root DIR] [--out profiles/gmt/batch_bench.json]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _import(root):
    sys.path.insert(0, root)
    import mpb200 as mp
    from mpb200 import _lib
    return mp, _lib


def _chunks(mask):
    chunks = np.zeros((len(mask) + 63) // 64 * 8, dtype=np.uint8)
    pk = np.packbits(mask, bitorder="little")
    chunks[:len(pk)] = pk
    return chunks.view(np.uint64)


def c2(mp, N=1_000_000):
    SS = mp.UnitHypercube(2)
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    return lambda: mp.MPProblem(SS, [0.1, 0.1], mp.BallGoal([0.9, 0.9], 0.01), CC), dict(N=N, seed=20240602)


def cars(mp, kind, N=200_000):
    rng = np.random.Generator(np.random.PCG64(20240605))
    V = np.column_stack([rng.random(N - 2), rng.random(N - 2), rng.uniform(0, 2 * np.pi, N - 2)])
    V = np.vstack([[0.1, 0.1, 0.0], V, [0.9, 0.9, 0.0]])
    SS = (mp.ReedsSheppMetricSpace if kind == "reedsshepp" else mp.DubinsQuasiMetricSpace)(0.01)
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    NNcls = mp.MetricNN if kind == "reedsshepp" else mp.QuasiMetricNN
    return lambda: mp.MPProblem(SS, V[0], mp.StateGoal(V[-1]), CC, V=NNcls(V, SS.dist, V[0])), dict(r=0.025)


def c4(mp, N=200_000):
    rng = np.random.Generator(np.random.PCG64(20240604))
    SS = mp.DoubleIntegrator(2)
    V = SS.lo + rng.random((N - 2, 4)) * (SS.hi - SS.lo)
    V = np.vstack([[0.1, 0.1, 0.0, 0.0], V, [0.9, 0.9, 0.0, 0.0]])
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    return lambda: mp.MPProblem(SS, V[0], mp.StateGoal(V[-1]), CC, V=mp.QuasiMetricNN(V, SS.dist, V[0])), dict(r=0.734)


class Roadmap:
    """the tables gmtstar(edge_checks=mode) left on the device and the calls that plan over them"""

    def __init__(self, mp, _lib, make, kw, mode):
        from mpb200.linearquadratic import LinearQuadratic
        from mpb200.simplecars import is_car_metric
        self.mp, self._lib, self.lib = mp, _lib, _lib.lib()
        self.P = P = make()
        mp.gmtstar(P, lam=1.0, edge_checks=mode, **kw)
        NN = self.NN = P.V
        self.N, self.r = len(NN), P.solution.metadata["r"]
        self.DF, self.DB = (NN.table, NN.table) if hasattr(NN, "table") else (NN.tableF, NN.tableB)
        self.edges = None
        if mode == "lazy":
            if is_car_metric(P.SS.dist):
                m = NN.dist.m
                self.edges = _lib.GmtEdges(_lib.GMT_EDGES_CAR, P.CC.handle(), None, 0.0, m.kind, m.r, m.s)
            elif isinstance(P.SS.dist, LinearQuadratic):
                self.edges = _lib.GmtEdges(_lib.GMT_EDGES_LQ, P.CC.handle(), NN.dist.handle(), NN.r, 0, 0.0, 0.0)
            else:
                self.edges = _lib.GmtEdges(_lib.GMT_EDGES_STRAIGHT, P.CC.handle(), None, 0.0, 0, 0.0, 0.0)

    def descs(self, queries):
        """one mpb200_gmt_desc per (init, goal chunks, lambda), all with the same space"""
        _lib = self._lib
        self.space = self.P.SS.desc()                 # arrays it points to live until the next desc() of the space
        sp = ctypes.pointer(self.space)
        return (_lib.GmtDesc * len(queries))(*[_lib.GmtDesc(self.DF.h, self.DB.h, _lib.ptr(c), i, lam * self.r, 1, sp)
                                               for i, c, lam in queries])

    def single(self, init, chunks, lam=1.0):
        """-> (device ms, outputs)"""
        _lib, N = self._lib, self.N
        d, res, path = self.descs([(init, chunks, lam)])[0], _lib.GmtResult(), np.empty(N, dtype=np.int64)
        segs = _lib.c_i64(0)
        if self.edges:
            rc = self.lib.mpb200_gmt_plan_lazy(self.NN.handle(), ctypes.byref(d), ctypes.byref(self.edges),
                                               ctypes.byref(res), ctypes.byref(segs), _lib.ptr(path), N, None, None)
        else:
            rc = self.lib.mpb200_gmt_plan(self.NN.handle(), ctypes.byref(d), ctypes.byref(res), _lib.ptr(path), N,
                                          None, None)
        _lib.check(rc)
        return self.lib.mpb200_last_ms_of(_lib.OP_PLAN, 1), _outputs(res, path, segs.value)

    def batch(self, queries):
        _lib, N, nq = self._lib, self.N, len(queries)
        ds = self.descs([(i, c, 1.0) for i, c in queries])
        res = (_lib.GmtResult * nq)()
        paths = np.empty((nq, N), dtype=np.int64)
        segs = np.zeros(nq, dtype=np.int64)
        _lib.check(self.lib.mpb200_gmt_plan_batch(self.NN.handle(), ds, nq,
                                                  ctypes.byref(self.edges) if self.edges else None, res,
                                                  _lib.ptr(segs), _lib.ptr(paths), N, None, None))
        return self.lib.mpb200_last_ms_of(_lib.OP_PLAN, 1), [_outputs(res[q], paths[q], segs[q]) for q in range(nq)]


def _outputs(res, path, segs):
    return (res.solved, res.goal, res.cost, res.iterations, res.expansions, res.checks, res.checks_in_bounds,
            res.path_len, path[:res.path_len].tobytes(), int(segs))


def scaling(mp, _lib, make, kw, mode, Qs, reps, seed):
    from mpb200.problems import goal_mask
    R = Roadmap(mp, _lib, make, kw, mode)
    V, SS = R.NN.V, R.P.SS
    F = np.unpackbits(R.NN.points_free(R.P.CC, SS).view(np.uint8), bitorder="little")[:R.N].astype(bool)
    free = np.flatnonzero(F)
    rng = np.random.Generator(np.random.PCG64(seed))
    qmax = max(Qs)
    inits = rng.choice(free, qmax) + 1
    centres = [V[j, :2].copy() for j in rng.choice(free, qmax)]
    goals = [_chunks(goal_mask(V, mp.BallGoal(c, 0.01), SS)) for c in centres]
    R.batch([(int(inits[0]), goals[0])])                                   # warm-up
    out = {}
    for Q in Qs:
        qs = [(int(inits[i]), goals[i]) for i in range(Q)]
        tb, ts = [], []
        for _ in range(reps):
            ms, ob = R.batch(qs)
            tb.append(ms)
            singles = [R.single(i, c) for i, c in qs]
            ts.append(sum(ms for ms, _ in singles))
            assert ob == [o for _, o in singles], "a query of the batch differs from its single plan"
        its = [o[3] for o in ob]
        out[str(Q)] = dict(batch_ms=statistics.median(tb), singles_sum_ms=statistics.median(ts),
                           speedup=statistics.median(ts) / statistics.median(tb), solved=sum(o[0] for o in ob),
                           iterations_max=max(its), iterations_mean=float(np.mean(its)),
                           batch_ms_all=tb, singles_sum_ms_all=ts, outputs_equal=True)
    out["grid_blocks_note"] = "occupancy-derived co-resident grid, the same for every Q"
    R.NN.close()
    return out, ([int(i) for i in inits[:qmax]], centres, ob)


def python_api(mp, make, kw, mode, inits, centres, ref):
    """gmtstar_batch(trees=False) from scratch on a fresh problem with the queries of the largest Q: its outputs equal
    the batch over the C ABI (same seeded samples); host wall time and the batch's device time"""
    import time
    P = make()
    t0 = time.perf_counter()
    sols = mp.gmtstar_batch(P, inits, [mp.BallGoal(c, 0.01) for c in centres], lam=1.0, edge_checks=mode,
                            trees=False, **kw)
    wall = time.perf_counter() - t0
    for s, o in zip(sols, ref):
        m = s.metadata
        assert (s.status == "solved", s.cost, m["iterations"], m["expansions"], m["checks"],
                np.asarray(m["path"], dtype=np.int64).tobytes()) == (bool(o[0]), o[2], o[3], o[4], o[5], o[8])
    P.V.close()
    return dict(Q=len(inits), from_scratch_s=wall, device_ms=sols[0].metadata["device_ms"], outputs_equal=True)


def q1_child(root, reps):
    """single-plan device times of the tree at `root` (runs in a child process)"""
    mp, _lib = _import(root)
    mp.init(0)
    out = {}
    for name, (make, kw), mode, lams in (("C2_table", c2(mp), "table", (0.5, 1.0, 2.0)),
                                         ("C2_lazy", c2(mp), "lazy", (1.0,)),
                                         ("RS_lazy", cars(mp, "reedsshepp"), "lazy", (1.0,)),
                                         ("DUB_lazy", cars(mp, "dubins"), "lazy", (1.0,)),
                                         ("C4_lazy", c4(mp), "lazy", (1.0,))):
        R = Roadmap(mp, _lib, make, kw, mode)
        from mpb200.problems import goal_mask
        chunks = _chunks(goal_mask(R.NN.V, R.P.goal, R.P.SS))
        for lam in lams:
            ms = [R.single(1, chunks, lam) for _ in range(reps + 1)]
            out["%s_lam%g" % (name, lam)] = dict(device_ms=statistics.median(m for m, _ in ms[1:]),
                                                 iterations=ms[-1][1][3], cost=ms[-1][1][2])
        R.NN.close()
    print("Q1JSON " + json.dumps(out))


def q1_compare(parent_root, rounds, reps):
    runs = {"parent": [], "this": []}
    for _ in range(rounds):
        for who, root in (("parent", parent_root), ("this", ROOT)):
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--q1-child", root, "--reps", str(reps)],
                               capture_output=True, text=True, cwd=ROOT)
            line = [l for l in p.stdout.splitlines() if l.startswith("Q1JSON ")]
            if p.returncode != 0 or not line:
                raise RuntimeError("q1 child (%s) failed:\n%s%s" % (who, p.stdout[-2000:], p.stderr[-4000:]))
            runs[who].append(json.loads(line[0][7:]))
    out = {}
    for k in runs["this"][0]:
        a = [r[k]["device_ms"] for r in runs["parent"]]
        b = [r[k]["device_ms"] for r in runs["this"]]
        assert all(r[k]["cost"] == runs["this"][0][k]["cost"] and r[k]["iterations"] == runs["this"][0][k]["iterations"]
                   for r in runs["parent"] + runs["this"]), k
        out[k] = dict(parent_ms=statistics.median(a), this_ms=statistics.median(b),
                      ratio=statistics.median(b) / statistics.median(a), parent_ms_all=a, this_ms_all=b,
                      iterations=runs["this"][0][k]["iterations"])
    return out


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
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--parent-root", default=None)
    ap.add_argument("--q1-child", default=None)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.q1_child:
        return q1_child(a.q1_child, a.reps)
    mp, _lib = _import(ROOT)
    mp.init(0)
    line = dict(gpu=gpu_info(),
                note="device ms = CUDA events around the planning kernel; medians of %d alternated repetitions" % a.reps)
    line["C2_scaling"] = {}
    for mode in ("table", "lazy"):
        line["C2_scaling"][mode], (inits, centres, ob) = scaling(mp, _lib, *c2(mp), mode, (1, 4, 16, 64), a.reps, 7)
        line["C2_scaling"][mode]["gmtstar_batch_trees_false"] = python_api(mp, *c2(mp), mode, inits, centres, ob)
    line["RS_lazy_scaling"] = scaling(mp, _lib, *cars(mp, "reedsshepp"), "lazy", (1, 4, 16, 64), a.reps, 8)[0]
    if a.parent_root:
        line["q1_vs_parent"] = q1_compare(os.path.abspath(a.parent_root), a.rounds, a.reps)
    line["gpu_after"] = gpu_info()
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
