#!/usr/bin/env python
"""A batch of PRM* queries over one roadmap (mpb200_sssp_plan_batch) against the same queries planned one by one
(mpb200_sssp_plan).

  scaling    C2 (2-D unit square, ISRR_2H, N = 1M free samples, seed 20240602, r = fmt_radius), the 64 random queries
             of scripts/gmt_batch_bench.py (free inits, BallGoal(radius 0.01) at free samples, seed 7), Q in
             {1, 4, 16, 64}; Reeds-Shepp and C4 (the N = 200k workloads of scripts/sssp_bench.py, seeds 8 and 9),
             Q in {1, 16, 64}.  Per Q, alternating the two, --reps times after a warm-up: the device time of the
             batch (CUDA events around its one launch) and the sum of the device times of the Q single plans;
             medians.  Rounds and levels of the queries (max, mean), the queries solved, and an assertion in every
             repetition that every query's outputs equal its single plan.
  yardstick  gmtstar_batch (table mode, trees=False) at lambda in {0.5, 1, 2} on the same 64 C2 queries and roadmap:
             GMT* cost over PRM* cost (min / median / max) over the queries both solve, and the queries PRM* solves
             that GMT* does not.
  q1         single PRM* plans of C2, RS and C4 (the problem's own query) in child processes that alternate this tree
             with --parent-root (a built checkout of the parent commit), --rounds times each: median device time of
             --reps re-plans over resident tables, and the spread.
The GPU's name and power limit are read in the same run.  Prints one JSON line; --out writes it to a file too.

  python scripts/sssp_batch_bench.py [--reps 5] [--parent-root DIR] [--out profiles/sssp/batch_bench.json]
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
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from gmt_batch_bench import _chunks, _import, c2, c4, cars, gpu_info  # noqa: E402


class Roadmap:
    """the tables prmstar left on the device and the PRM* calls that plan over them"""

    def __init__(self, mp, _lib, make, kw):
        self.mp, self._lib, self.lib = mp, _lib, _lib.lib()
        self.P = P = make()
        mp.prmstar(P, **kw)
        NN = self.NN = P.V
        self.N = len(NN)
        self.DF, self.DB = (NN.table, NN.table) if hasattr(NN, "table") else (NN.tableF, NN.tableB)

    def descs(self, queries):
        _lib = self._lib
        return (_lib.GmtDesc * len(queries))(*[_lib.GmtDesc(self.DF.h, self.DB.h, _lib.ptr(c), i, 0.0, 1, None)
                                               for i, c in queries])

    def single(self, init, chunks):
        """-> (device ms, outputs)"""
        _lib, N = self._lib, self.N
        d, res, path = self.descs([(init, chunks)])[0], _lib.SsspResult(), np.empty(N, dtype=np.int64)
        _lib.check(self.lib.mpb200_sssp_plan(self.NN.handle(), ctypes.byref(d), ctypes.byref(res), _lib.ptr(path), N,
                                             None, None))
        return self.lib.mpb200_last_ms_of(_lib.OP_PLAN, 0), _outputs(res, path)

    def batch(self, queries):
        _lib, N, nq = self._lib, self.N, len(queries)
        ds = self.descs(queries)
        res = (_lib.SsspResult * nq)()
        paths = np.empty((nq, N), dtype=np.int64)
        _lib.check(self.lib.mpb200_sssp_plan_batch(self.NN.handle(), ds, nq, res, _lib.ptr(paths), N, None, None))
        return self.lib.mpb200_last_ms_of(_lib.OP_PLAN, 0), [_outputs(res[q], paths[q]) for q in range(nq)]


def _outputs(res, path):
    return (res.solved, res.goal, res.cost, res.path_len, res.rounds, res.levels, res.reached,
            path[:res.path_len].tobytes())


def queries(mp, R, qmax, seed):
    """the queries of gmt_batch_bench.scaling: free inits, BallGoal(0.01) around free samples' positions"""
    from mpb200.problems import goal_mask
    V, SS = R.NN.V, R.P.SS
    F = np.unpackbits(R.NN.points_free(R.P.CC, SS).view(np.uint8), bitorder="little")[:R.N].astype(bool)
    free = np.flatnonzero(F)
    rng = np.random.Generator(np.random.PCG64(seed))
    inits = rng.choice(free, qmax) + 1
    centres = [V[j, :2].copy() for j in rng.choice(free, qmax)]
    return [int(i) for i in inits], centres, [_chunks(goal_mask(V, mp.BallGoal(c, 0.01), SS)) for c in centres]


def scaling(mp, _lib, make, kw, Qs, reps, seed, yardstick=False):
    R = Roadmap(mp, _lib, make, kw)
    inits, centres, goals = queries(mp, R, max(Qs), seed)
    R.batch([(inits[0], goals[0])])                                        # warm-up
    R.single(inits[0], goals[0])
    out = {}
    for Q in Qs:
        qs = list(zip(inits[:Q], goals[:Q]))
        tb, ts = [], []
        for _ in range(reps):
            ms, ob = R.batch(qs)
            tb.append(ms)
            singles = [R.single(i, c) for i, c in qs]
            ts.append(sum(ms for ms, _ in singles))
            assert ob == [o for _, o in singles], "a query of the batch differs from its single plan"
        rounds, levels = [o[4] for o in ob], [o[5] for o in ob]
        out[str(Q)] = dict(batch_ms=statistics.median(tb), singles_sum_ms=statistics.median(ts),
                           speedup=statistics.median(ts) / statistics.median(tb), solved=sum(o[0] for o in ob),
                           rounds_max=max(rounds), rounds_mean=float(np.mean(rounds)), levels_max=max(levels),
                           levels_mean=float(np.mean(levels)), batch_ms_all=tb, singles_sum_ms_all=ts,
                           outputs_equal=True)
    out["grid_blocks_note"] = "occupancy-derived co-resident grid, the same for every Q"
    if yardstick:
        out["yardstick"] = gmt_yardstick(mp, R, kw, inits, centres, ob)
    R.NN.close()
    return out


def gmt_yardstick(mp, R, kw, inits, centres, prm):
    """gmtstar_batch over the same problem (its tables rebuilt identically) and queries: GMT* cost / PRM* cost"""
    out = {}
    for lam in (0.5, 1.0, 2.0):
        sols = mp.gmtstar_batch(R.P, inits, [mp.BallGoal(c, 0.01) for c in centres], lam=lam, trees=False, **kw)
        ratios, prm_only = [], 0
        for s, o in zip(sols, prm):
            if s.status == "solved":
                assert o[0] and o[2] <= s.cost
                ratios.append(s.cost / o[2] if o[2] > 0 else 1.0)   # an init inside its goal costs 0 in both
            elif o[0]:
                prm_only += 1
        out[str(lam)] = dict(both_solved=len(ratios), ratio_min=min(ratios), ratio_median=statistics.median(ratios),
                             ratio_max=max(ratios), prm_solves_gmt_does_not=prm_only)
    return out


def q1_child(root, reps):
    """single PRM* plan device times of the tree at `root` (runs in a child process)"""
    mp, _lib = _import(root)
    mp.init(0)
    out = {}
    for name, (make, kw) in (("C2", c2(mp)), ("RS", cars(mp, "reedsshepp")), ("C4", c4(mp))):
        P = make()
        mp.prmstar(P, **kw)
        NN = P.V
        DF, DB = (NN.table, NN.table) if hasattr(NN, "table") else (NN.tableF, NN.tableB)
        from mpb200.problems import goal_mask
        chunks = _chunks(goal_mask(NN.V, P.goal, P.SS))
        N = len(NN)
        path = np.empty(N, dtype=np.int64)
        ms = []
        for _ in range(reps + 1):
            d, res = _lib.GmtDesc(DF.h, DB.h, _lib.ptr(chunks), 1, 0.0, 1, None), _lib.SsspResult()
            _lib.check(_lib.lib().mpb200_sssp_plan(NN.handle(), ctypes.byref(d), ctypes.byref(res), _lib.ptr(path),
                                                   N, None, None))
            ms.append(_lib.lib().mpb200_last_ms_of(_lib.OP_PLAN, 0))
        out[name] = dict(device_ms=statistics.median(ms[1:]), rounds=res.rounds, levels=res.levels, cost=res.cost,
                         path=path[:res.path_len].tolist())
        NN.close()
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
    ref = runs["parent"][0]
    for k in ref:
        for r in runs["parent"] + runs["this"]:          # the same plan from both trees
            assert all(r[k][f] == ref[k][f] for f in ("rounds", "levels", "cost", "path")), k
        a = [r[k]["device_ms"] for r in runs["parent"]]
        b = [r[k]["device_ms"] for r in runs["this"]]
        out[k] = dict(parent_ms=statistics.median(a), this_ms=statistics.median(b),
                      ratio=statistics.median(b) / statistics.median(a), parent_ms_all=a, this_ms_all=b,
                      spread_parent=(max(a) - min(a)) / statistics.median(a),
                      spread_this=(max(b) - min(b)) / statistics.median(b),
                      rounds=ref[k]["rounds"], levels=ref[k]["levels"])
    return out


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
                note="device ms = CUDA events around the one cooperative launch of each call (MPB200_OP_PLAN); "
                     "medians of %d alternated repetitions after a warm-up" % a.reps)
    line["C2_scaling"] = scaling(mp, _lib, *c2(mp), (1, 4, 16, 64), a.reps, 7, yardstick=True)
    line["RS_scaling"] = scaling(mp, _lib, *cars(mp, "reedsshepp"), (1, 16, 64), a.reps, 8)
    line["C4_scaling"] = scaling(mp, _lib, *c4(mp), (1, 16, 64), a.reps, 9)
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
