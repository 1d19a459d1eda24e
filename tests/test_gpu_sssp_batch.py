"""A batch of PRM* queries over one roadmap (mpb200_sssp_plan_batch, planners.prmstar_batch): every query's outputs,
rounds, levels and |R| included, equal the single plan of that query (mpb200_sssp_plan) byte for byte, and all but the
round count equal tests/oracle_sssp.py, on the eight problem kinds of test_gpu_gmt.py and the duplicated-sample and
lattice sets of test_gpu_sssp.py, with and without checkpts; a query's outputs do not depend on the rest of its batch,
its order or the grid size; one launch per batch; rows that do not fit path_cap stay untouched; prmstar_batch of
(1, P.goal) is prmstar; PRM* dominates GMT* query by query; the argument checks of the C ABI; C2 at full size."""
import ctypes
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest

from oracle_sssp import sssp_numpy, sssp_oracle
from test_gpu_gmt import CASES, _case, _tables_of, fx_bits
from test_gpu_sssp import _tie_sets

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EARG, ENOMEM = -1, -4


def _chunks(mask):
    chunks = np.zeros((len(mask) + 63) // 64 * 8, dtype=np.uint8)
    pk = np.packbits(mask, bitorder="little")
    chunks[:len(pk)] = pk
    return chunks.view(np.uint64)


def _make(mp, orc, name):
    return _tie_sets(mp, name) if name in ("duplicates", "lattice") else _case(mp, orc, name)


class Roadmap:
    """the tables, edge bits and point bits prmstar left on the device, fetched too, and the C calls over them"""

    def __init__(self, mp, orc, name, P=None, kw=None):
        from mpb200 import _lib
        from mpb200.problems import goal_mask
        if P is None:
            make, kw = _make(mp, orc, name)
            P = make()
            mp.prmstar(P, **kw)
        self.P, self.NN = P, P.V
        NN = P.V
        self.N = N = len(NN)
        if kw.get("connections") == "K":
            self.DF, self.DB = (NN.table_mknn, NN.table_knn) if hasattr(NN, "table_knn") else (NN.table_mknnF,
                                                                                              NN.table_knnB)
        elif hasattr(NN, "tableF"):
            self.DF, self.DB = NN.tableF, NN.tableB
        else:
            self.DF = self.DB = NN.table
        self.name, self.kw = name, kw
        self.free = fx_bits(NN.points_free(P.CC, P.SS), N)
        self.goal = goal_mask(NN.V, P.goal, P.SS)
        self.lib = _lib.lib()
        self._tables = None

    def tables(self):
        if self._tables is None:
            self._tables = _tables_of(self.NN, self.name, self.kw)
        return self._tables

    def oracle(self, query, checkpts):
        _, B, ebits = self.tables()
        free = self.free if checkpts else np.ones(self.N, dtype=bool)
        return sssp_oracle(self.N, B.colptr, B.rowval, B.nzval, ebits, free, query[1], init=query[0])

    def queries(self, checkpts, seed=5):
        """the problem's own query, six free inits with one-state goals, an init in its own goal, an empty goal mask,
        an unreachable goal (when the roadmap has one from that init) and a duplicate"""
        N = self.N
        free = np.flatnonzero(self.free)
        rng = np.random.Generator(np.random.PCG64(seed))
        one = lambda j: np.arange(N) == j
        q = [(1, self.goal)]
        for _ in range(6):
            a, b = rng.choice(free, 2, replace=False)
            q.append((int(a) + 1, one(int(b))))
        j = int(rng.choice(free))
        q.append((j + 1, one(j)))
        e0 = int(rng.choice(free))
        q.append((e0 + 1, np.zeros(N, dtype=bool)))
        tree = self.oracle(q[-1], checkpts)
        far = np.flatnonzero(~np.isfinite(tree["costs"]))
        if far.size:
            q.append((e0 + 1, one(int(rng.choice(far)))))
        q.append(q[2])
        return q, bool(far.size)

    def descs(self, queries, checkpts=1):
        from mpb200 import _lib
        self._keep = [_chunks(m) for _, m in queries]
        ds = (_lib.GmtDesc * len(queries))()
        for i, (init, _) in enumerate(queries):
            ds[i] = _lib.GmtDesc(self.DF.h, self.DB.h, _lib.ptr(self._keep[i]), init, 0.0, checkpts, None)
        return ds

    def batch(self, queries, checkpts=1, path_cap=None, trees=True):
        """mpb200_sssp_plan_batch -> (rc, per-query outputs, results)"""
        from mpb200 import _lib
        nq, N = len(queries), self.N
        cap = N if path_cap is None else path_cap
        ds = self.descs(queries, checkpts)
        res = (_lib.SsspResult * nq)()
        paths = np.full((nq, max(cap, 1)), -7, dtype=np.int64)
        T = np.full((nq, N), -7, dtype=np.int64) if trees else None
        C = np.full((nq, N), -7.0) if trees else None
        rc = self.lib.mpb200_sssp_plan_batch(self.NN.handle(), ds, nq, res, _lib.ptr(paths), cap, _lib.ptr(T),
                                             _lib.ptr(C))
        return rc, [self._out(res[i], paths[i], None if T is None else T[i], None if C is None else C[i])
                    for i in range(nq)], res

    def single(self, query, checkpts=1):
        """mpb200_sssp_plan of one query -> (rc, outputs)"""
        from mpb200 import _lib
        N = self.N
        ds = self.descs([query], checkpts)
        res = _lib.SsspResult()
        path = np.full(N, -7, dtype=np.int64)
        T, C = np.full(N, -7, dtype=np.int64), np.full(N, -7.0)
        rc = self.lib.mpb200_sssp_plan(self.NN.handle(), ds, ctypes.byref(res), _lib.ptr(path), N, _lib.ptr(T),
                                       _lib.ptr(C))
        return rc, self._out(res, path, T, C)

    @staticmethod
    def _out(res, path, T, C):
        n = res.path_len
        return (res.solved, res.goal, np.float64(res.cost).tobytes(), n, res.rounds, res.levels, res.reached,
                path[:n].tobytes() if n <= len(path) else None, None if T is None else T.tobytes(),
                None if C is None else C.tobytes())

    def close(self):
        self.NN.close()


def _equals_oracle(out, ref):
    solved, goal, cost, n, _, levels, reached, path, T, C = out
    assert bool(solved) == ref["solved"] and goal == ref["goal"]
    assert cost == np.float64(ref["cost"]).tobytes()
    assert n == len(ref["path"]) and path == np.asarray(ref["path"], dtype=np.int64).tobytes()
    assert T == ref["tree"].astype(np.int64).tobytes() and C == ref["costs"].tobytes()
    assert (levels, reached) == (ref["levels"], ref["reached"])


@pytest.mark.parametrize("name", CASES + ["duplicates", "lattice"])
def test_batch_equals_single_plans_and_the_oracle(gpu, orc, name):
    mp = gpu
    R = Roadmap(mp, orc, name)
    for checkpts in (1, 0):
        qs, has_far = R.queries(checkpts)
        rc, outs, res = R.batch(qs, checkpts)
        assert rc == 0, R.lib.mpb200_last_error()
        for i, q in enumerate(qs):
            rc1, one = R.single(q, checkpts)
            assert rc1 == 0 and outs[i] == one, (checkpts, i)
            assert res[i].grid_blocks == res[0].grid_blocks
            _equals_oracle(outs[i], R.oracle(q, checkpts))
        assert outs[0][0] == 1                                            # the problem's own query is solved
        init_in_goal, empty = outs[7], outs[8]
        assert init_in_goal[0] == 1 and init_in_goal[3] == 1 and init_in_goal[2] == np.float64(0.0).tobytes()
        assert empty[0] == 0 and empty[3] == 0 and empty[6] > 0
        if has_far:
            assert outs[9][0] == 0                                        # the unreachable goal fails
        assert outs[-1] == outs[2]
    if name == "duplicates":
        assert has_far                                                    # non-free samples under checkpts
    R.close()


def _batch_outputs(mp, orc, name):
    R = Roadmap(mp, orc, name)
    qs, _ = R.queries(1)
    rc, outs, res = R.batch(qs)
    assert rc == 0, R.lib.mpb200_last_error()
    R.close()
    return outs, res[0].grid_blocks


def test_outputs_do_not_depend_on_the_rest_of_the_batch_or_the_grid(gpu, orc, tmp_path):
    mp = gpu
    R = Roadmap(mp, orc, "2d_20k")
    qs, _ = R.queries(1)
    rc, base, res = R.batch(qs)
    assert rc == 0
    blocks = res[0].grid_blocks
    perm = np.random.Generator(np.random.PCG64(3)).permutation(len(qs))
    rc, outs, _ = R.batch([qs[i] for i in perm])
    assert rc == 0 and [outs[k] for k in np.argsort(perm)] == base
    h = len(qs) // 2
    rc1, first, _ = R.batch(qs[:h])
    rc2, second, _ = R.batch(qs[h:])
    assert rc1 == rc2 == 0 and first + second == base
    for i, q in enumerate(qs):
        rc, alone, _ = R.batch([q])
        assert rc == 0 and alone == [base[i]], i
    R.close()
    dump = str(tmp_path / "sssp_batch_child.pkl")
    code = ("import sys, pickle; sys.path[:0] = [%r, %r]; import mpb200 as mp; mp.init(0)\n"
            "from oracle import oracle as orc; orc.lib()\n"
            "import test_gpu_sssp_batch as t\n"
            "o = t._batch_outputs(mp, orc, '2d_20k')\n"
            "pickle.dump(o, open(%r, 'wb'))\n" % (ROOT, os.path.join(ROOT, "tests"), dump))
    subprocess.run([sys.executable, "-c", code], check=True, env=dict(os.environ, MPB200_GMT_GRID="37"), cwd=ROOT)
    with open(dump, "rb") as f:
        c, blocks37 = pickle.load(f)
    assert blocks37 == 37 != blocks and c == base


def test_one_launch_per_batch_and_rows_past_path_cap_untouched(gpu, orc):
    mp = gpu
    R = Roadmap(mp, orc, "2d_20k")
    qs, _ = R.queries(1)
    before = R.lib.mpb200_launch_count()
    rc, full, _ = R.batch(qs)
    assert rc == 0 and R.lib.mpb200_launch_count() - before == 1
    lens = sorted({o[3] for o in full if o[3] > 1})
    assert len(lens) >= 2
    cap = lens[len(lens) // 2] - 1                                        # some rows fit, some do not
    from mpb200 import _lib
    ds = R.descs(qs)
    res = (_lib.SsspResult * len(qs))()
    paths = np.full((len(qs), cap), -7, dtype=np.int64)
    before = R.lib.mpb200_launch_count()
    assert R.lib.mpb200_sssp_plan_batch(R.NN.handle(), ds, len(qs), res, _lib.ptr(paths), cap, None, None) == 0
    assert R.lib.mpb200_launch_count() - before == 1
    fit = 0
    for i, o in enumerate(full):
        assert R._out(res[i], np.zeros(0, np.int64), None, None)[:7] == o[:7]
        if o[3] <= cap:
            fit += 1
            assert paths[i, :o[3]].tobytes() == o[7] and np.all(paths[i, o[3]:] == -7)
        else:
            assert np.all(paths[i] == -7), i
    assert 0 < fit < len(qs)
    R.close()


def _comparable(sol):
    m = dict(sol.metadata)
    for key in ("device_ms", "query", "batch_size"):
        m.pop(key, None)
    return sol.status, np.float64(sol.cost).tobytes(), {k: (v.tobytes() if isinstance(v, np.ndarray) else v)
                                                        for k, v in m.items()}


def _uniform_set(mp):
    """2-D samples drawn uniformly among boxes, so some lie inside an obstacle"""
    import fixtures as fx
    SS = mp.UnitHypercube(2)
    CC = mp.PointRobotNDBoxes([mp.BoxBounds(b) for b in fx.BOXES2D])
    V = np.random.Generator(np.random.PCG64(8)).random((3000, 2))
    V = np.vstack([[0.1, 0.1], V, [0.9, 0.9]])
    return lambda: mp.MPProblem(SS, V[0], mp.PointGoal(V[-1]), CC, V=mp.MetricNN(V, SS.dist, V[0])), dict(r=0.05)


def test_python_api(gpu):
    mp = gpu
    make, kw = _uniform_set(mp)
    Pp, Pb = make(), make()
    mp.prmstar(Pp, **kw)
    sols = mp.prmstar_batch(Pb, [1], [Pb.goal], **kw)
    assert len(sols) == 1 and sols[0].metadata["query"] == 0 and sols[0].metadata["batch_size"] == 1
    assert set(sols[0].metadata) == set(Pp.solution.metadata) | {"query", "batch_size"}
    assert _comparable(sols[0]) == _comparable(Pp.solution) and Pp.status == "solved"
    assert sols[0].metadata["device_ms"] > 0
    nonfree = int(np.flatnonzero(~fx_bits(Pp.V.points_free(Pp.CC, Pp.SS), len(Pp.V)))[0]) + 1
    lib = mp.load()
    P1, P2 = make(), make()
    before = lib.mpb200_launch_count()
    mp.prmstar_batch(P1, [1], [P1.goal], **kw)
    one = lib.mpb200_launch_count() - before
    before = lib.mpb200_launch_count()
    two = mp.prmstar_batch(P2, [1, nonfree], [P2.goal, P2.goal], **kw)
    assert lib.mpb200_launch_count() - before == one                      # no launch for the non-free init
    assert two[1].status == "failed" and two[1].metadata == {"query": 1, "batch_size": 2}
    assert _comparable(two[0]) == _comparable(sols[0]) and two[0].metadata["batch_size"] == 2
    light = mp.prmstar_batch(make(), [1], [Pb.goal], trees=False, **kw)[0]
    assert light.metadata["tree"] is None and light.metadata["costs"] is None and light.metadata["cumcost"] is None
    assert light.metadata["path"] == sols[0].metadata["path"] and light.cost == sols[0].cost
    for P in (Pp, Pb, P1, P2):
        P.V.close()


def test_prm_batch_dominates_gmt_batch_and_shortcutting_never_raises_a_cost(gpu, orc):
    mp = gpu
    make, kw = _case(mp, orc, "2d_20k")
    P = make()
    mp.prmstar(P, **kw)
    N = len(P.V)
    free = np.flatnonzero(fx_bits(P.V.points_free(P.CC, P.SS), N))
    rng = np.random.Generator(np.random.PCG64(17))
    inits = [1] + [int(i) + 1 for i in rng.choice(free, 8, replace=False)]
    goals = [P.goal] + [mp.StateGoal(P.V.V[int(j)]) for j in rng.choice(free, 8, replace=False)]
    prm = mp.prmstar_batch(P, inits, goals, **kw)
    assert prm[0].status == "solved"
    for lam in (0.0, 1.0, 4.0):
        gmt = mp.gmtstar_batch(P, inits, goals, lam=lam, **kw)
        for q, (p, g) in enumerate(zip(prm, gmt)):
            if g.status == "solved":
                assert p.status == "solved" and p.cost <= g.cost, (lam, q)
    solved = [p for p in prm if p.status == "solved" and len(p.metadata["path"]) > 1]
    out = mp.shortcut_paths(P, [p.metadata["path"] for p in solved], subdivisions=4)
    assert len(out) == len(solved) > 1
    for o, p in zip(out, solved):
        assert o["cost"] <= p.cost
    P.V.close()


def test_batch_argument_checks(gpu, orc):
    mp = gpu
    from mpb200 import _lib
    R = Roadmap(mp, orc, "2d_2k")
    qs = R.queries(1)[0][:4]
    lib, NN = R.lib, R.NN
    other = mp.MetricNN(NN.V.copy())                                      # a table of another sample set
    other.build_table_checked(0.05, R.P.CC, R.P.SS)
    fresh = mp.MetricNN(NN.V.copy())                                      # no point bits: checkpts is rejected
    fresh.build_table_checked(0.05, R.P.CC, R.P.SS)
    launches = lib.mpb200_launch_count()

    def rejects(code, ds=None, nq=None, res=True, paths=True, cap=None):
        ds = R.descs(qs) if ds is None else ds
        n = len(qs) if nq is None else nq
        rs = (_lib.SsspResult * max(n, 1))() if res else None
        cap = R.N if cap is None else cap
        p = np.empty((max(n, 1), max(cap, 1)), dtype=np.int64) if paths else None
        return lib.mpb200_sssp_plan_batch(NN.handle(), ds, n, rs, _lib.ptr(p), cap, None, None) == code

    assert rejects(EARG, nq=0) and rejects(EARG, nq=-3)
    assert lib.mpb200_sssp_plan_batch(NN.handle(), None, 2, (_lib.SsspResult * 2)(), None, 0, None, None) == EARG
    assert rejects(EARG, res=False)                                       # NULL res
    assert rejects(EARG, paths=False)                                     # NULL paths, path_cap > 0
    assert rejects(EARG, cap=-1)
    for field, bad in (("init", 0), ("init", R.N + 1), ("goal_bits", None)):
        ds = R.descs(qs)
        setattr(ds[2], field, bad)                                        # one bad query among good ones
        assert rejects(EARG, ds=ds), field
    for field, value in (("fwd", other.table.h), ("bwd", other.table.h), ("checkpts", 0), ("fwd", None)):
        ds = R.descs(qs)
        setattr(ds[3], field, value)                                      # shared fields that differ
        assert rejects(EARG, ds=ds), field
    for field in ("fwd", "bwd"):
        ds = R.descs(qs)
        for i in range(len(qs)):
            setattr(ds[i], field, other.table.h)                          # all alike, but of another set
        assert rejects(EARG, ds=ds), field
    ds = R.descs(qs)
    for i in range(len(qs)):
        ds[i].fwd = ds[i].bwd = fresh.table.h
    assert lib.mpb200_sssp_plan_batch(fresh.handle(), ds, len(qs), (_lib.SsspResult * len(qs))(), None, 0, None,
                                      None) == EARG
    import torch
    total = torch.cuda.get_device_properties(0).total_memory
    nq = total // (52 * R.N) + 1                                          # scratch > device memory
    one = R.descs(qs[:1])[0]
    ds = (_lib.GmtDesc * nq)(*([one] * nq))
    rs = (_lib.SsspResult * nq)()
    assert lib.mpb200_sssp_plan_batch(NN.handle(), ds, nq, rs, None, 0, None, None) == ENOMEM
    assert lib.mpb200_launch_count() == launches                          # no rejection launched
    rc, _, _ = R.batch(qs)
    assert rc == 0 and lib.mpb200_launch_count() == launches + 1
    fresh.close()
    other.close()
    R.close()


def test_batch_full_size_c2_equals_single_plans_and_the_numpy_restatement(gpu):
    """C2 (ISRR_2H, N = 1M, r from fmt_radius): 16 random queries in one batch"""
    mp = gpu
    from mpb200.problems import goal_mask
    N = 1_000_000
    SS = mp.UnitHypercube(2)
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    P = mp.MPProblem(SS, [0.1, 0.1], mp.BallGoal([0.9, 0.9], 0.01), CC)
    st, _, _ = mp.prmstar(P, N, seed=20240602)
    assert st == "solved"
    R = Roadmap(mp, None, "c2", P=P, kw={})
    free = np.flatnonzero(R.free)
    rng = np.random.Generator(np.random.PCG64(2024))
    qs = [(int(a) + 1, goal_mask(P.V.V, mp.BallGoal(P.V.V[int(b)], 0.01), SS))
          for a, b in zip(rng.choice(free, 16), rng.choice(free, 16))]
    rc, outs, _ = R.batch(qs)
    assert rc == 0 and sum(o[0] for o in outs) > 0
    for i, q in enumerate(qs):
        rc1, one = R.single(q)
        assert rc1 == 0 and outs[i] == one, i
    T = P.V.fetch_table(P.V.table)
    from mpb200 import _lib
    bits = np.empty((T.nnz + 63) // 64, dtype=np.uint64)
    _lib.check(_lib.lib().mpb200_table_fetch_edge_bits(P.V.table.h, _lib.ptr(bits)))
    ebits = fx_bits(bits, T.nnz)
    for i in (0, 1):
        ref = sssp_numpy(N, T.colptr, T.rowval, T.nzval, ebits, R.free, qs[i][1], init=qs[i][0])
        _equals_oracle(outs[i], ref)
    R.close()
