"""A batch of GMT* queries over one roadmap (mpb200_gmt_plan_batch, planners.gmtstar_batch): every query's outputs equal
the single plan of that query over the same tables, byte for byte, in table and lazy mode on every problem kind;
gmtstar_batch of (1, P.goal) is gmtstar; queries from other inits equal tests/oracle_gmt.py; a query's outputs do not
depend on the rest of its batch, the run or the grid size; one launch per batch; the argument checks of the C ABI;
C2 at full size."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle_gmt import gmt_oracle
from test_gpu_gmt import CASES, _case, fx_bits
from test_gpu_gmt_lazy import EXTRA, _fetch_tables, _setup

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EARG, ENOMEM = -1, -4
LAMS = (0.0, 0.25, 1.0, 4.0)


def _chunks(mask):
    chunks = np.zeros((len(mask) + 63) // 64 * 8, dtype=np.uint8)
    pk = np.packbits(mask, bitorder="little")
    chunks[:len(pk)] = pk
    return chunks.view(np.uint64)


class Roadmap:
    """the tables, bits and edge test gmtstar(edge_checks=mode) left on the device, with a mixed set of queries"""

    def __init__(self, mp, orc, name, mode, lam=1.0, seed=5):
        from mpb200 import _lib
        from mpb200.problems import goal_mask
        from mpb200.planners import _gmt_edges
        from mpb200.linearquadratic import LinearQuadratic
        from mpb200.simplecars import is_car_metric
        make, kw, _ = _setup(mp, orc, name)
        self.P = P = make()
        mp.gmtstar(P, lam=lam, edge_checks=mode, **kw)
        self.NN = NN = P.V
        self.N = N = len(NN)
        self.r = P.solution.metadata["r"]
        if kw.get("connections") == "K":
            self.DF, self.DB = (NN.table_mknn, NN.table_knn) if hasattr(NN, "table_knn") else (NN.table_mknnF,
                                                                                              NN.table_knnB)
        elif hasattr(NN, "tableF"):
            self.DF, self.DB = NN.tableF, NN.tableB
        else:
            self.DF = self.DB = NN.table
        rm = dict(NN=NN, car=is_car_metric(P.SS.dist), lq=isinstance(P.SS.dist, LinearQuadratic))
        self.edges = _gmt_edges(rm, P.CC) if mode == "lazy" else None
        free = np.flatnonzero(fx_bits(NN.points_free(P.CC, P.SS), N))
        rng = np.random.Generator(np.random.PCG64(seed))
        one = lambda j: np.arange(N) == j
        q = [(1, goal_mask(NN.V, P.goal, P.SS), lam)]                     # the problem's own query
        for i in range(6):                                                 # other inits and state goals
            a, b = rng.choice(free, 2, replace=False)
            q.append((int(a) + 1, one(b), LAMS[i % 4]))
        j = int(rng.choice(free))
        q.append((j + 1, one(j), 1.0))                                     # init in its own goal
        q.append((int(rng.choice(free)) + 1, np.zeros(N, dtype=bool), 1.0))  # empty goal mask
        q.append(q[2])                                                     # a duplicate
        self.queries = q
        self.lib = _lib.lib()

    def descs(self, queries, checkpts=1):
        from mpb200 import _lib
        self.space = self.P.SS.desc()                 # arrays it points to live until the next desc() of the space
        self._keep = [_chunks(m) for _, m, _ in queries]
        ds = (_lib.GmtDesc * len(queries))()
        for i, (init, _, lam) in enumerate(queries):
            ds[i] = _lib.GmtDesc(self.DF.h, self.DB.h, _lib.ptr(self._keep[i]), init, lam * self.r, checkpts,
                                 ctypes.pointer(self.space))
        return ds

    def batch(self, queries, path_cap=None, trees=True, descs=None):
        """mpb200_gmt_plan_batch -> (rc, per-query outputs)"""
        from mpb200 import _lib
        nq, N = len(queries), self.N
        cap = N if path_cap is None else path_cap
        ds = self.descs(queries) if descs is None else descs
        res = (_lib.GmtResult * nq)()
        paths = np.full((nq, max(cap, 1)), -7, dtype=np.int64)
        T = np.empty((nq, N), dtype=np.int64) if trees else None
        C = np.empty((nq, N)) if trees else None
        segs = np.full(nq, -1, dtype=np.int64)
        rc = self.lib.mpb200_gmt_plan_batch(self.NN.handle(), ds, nq, ctypes.byref(self.edges) if self.edges else None,
                                            res, _lib.ptr(segs), _lib.ptr(paths), cap, _lib.ptr(T), _lib.ptr(C))
        return rc, [self._out(res[i], paths[i], None if T is None else T[i], None if C is None else C[i],
                              segs[i] if self.edges else None) for i in range(nq)], res

    def single(self, query):
        """mpb200_gmt_plan / _lazy of one query -> (rc, outputs)"""
        from mpb200 import _lib
        N = self.N
        ds = self.descs([query])
        res = _lib.GmtResult()
        path = np.full(N, -7, dtype=np.int64)
        T, C = np.empty(N, dtype=np.int64), np.empty(N)
        segs = _lib.c_i64(-1)
        if self.edges:
            rc = self.lib.mpb200_gmt_plan_lazy(self.NN.handle(), ds, ctypes.byref(self.edges), ctypes.byref(res),
                                               ctypes.byref(segs), _lib.ptr(path), N, _lib.ptr(T), _lib.ptr(C))
        else:
            rc = self.lib.mpb200_gmt_plan(self.NN.handle(), ds, ctypes.byref(res), _lib.ptr(path), N, _lib.ptr(T),
                                          _lib.ptr(C))
        return rc, self._out(res, path, T, C, segs.value if self.edges else None), res

    @staticmethod
    def _out(res, path, T, C, segs):
        n = res.path_len
        return (res.solved, res.goal, np.float64(res.cost).tobytes(), res.iterations, res.expansions, res.checks,
                res.checks_in_bounds, n, path[:n].tobytes() if n <= len(path) else None,
                None if T is None else T.tobytes(), None if C is None else C.tobytes(), segs)

    def close(self):
        self.NN.close()


@pytest.mark.parametrize("mode", ["table", "lazy"])
@pytest.mark.parametrize("name", CASES + EXTRA)
def test_batch_equals_single_plans(gpu, orc, name, mode):
    mp = gpu
    R = Roadmap(mp, orc, name, mode)
    rc, outs, res = R.batch(R.queries)
    assert rc == 0, R.lib.mpb200_last_error()
    for i, q in enumerate(R.queries):
        rc1, one, r1 = R.single(q)
        assert rc1 == 0 and outs[i] == one, i
        assert res[i].grid_blocks == res[0].grid_blocks
    # (1, P.goal) is gmtstar's plan; an init in its goal is solved at iteration 0; an empty goal mask fails
    assert outs[0][0] == (R.P.status == "solved")
    init_in_goal, empty = outs[7], outs[8]
    assert init_in_goal[0] == 1 and init_in_goal[3] == 0 and init_in_goal[7] == 1 and init_in_goal[5] == 0
    assert empty[0] == 0 and empty[7] == 0 and empty[3] > 0
    assert outs[9] == outs[2]
    R.close()


def _comparable(sol):
    m = dict(sol.metadata)
    for key in ("device_ms", "query", "batch_size"):
        m.pop(key, None)
    return sol.status, np.float64(sol.cost).tobytes(), {k: (v.tobytes() if isinstance(v, np.ndarray) else v)
                                                        for k, v in m.items()}


@pytest.mark.parametrize("mode", ["table", "lazy"])
@pytest.mark.parametrize("name", ["2d_20k", "reedsshepp"])
def test_query_one_is_gmtstar(gpu, orc, name, mode):
    mp = gpu
    make, kw = _case(mp, orc, name)
    Pg, Pb = make(), make()
    mp.gmtstar(Pg, lam=1.0, edge_checks=mode, **kw)
    sols = mp.gmtstar_batch(Pb, [1], [Pb.goal], lam=1.0, edge_checks=mode, **kw)
    assert len(sols) == 1 and sols[0].metadata["query"] == 0 and sols[0].metadata["batch_size"] == 1
    assert set(sols[0].metadata) == set(Pg.solution.metadata) | {"query", "batch_size"}
    assert _comparable(sols[0]) == _comparable(Pg.solution) and Pg.status == "solved"
    assert sols[0].metadata["device_ms"] > 0
    Pg.V.close(); Pb.V.close()


@pytest.mark.parametrize("name", ["2d_2k", "dubins"])
def test_batch_equals_the_oracle_from_other_inits(gpu, orc, name):
    mp = gpu
    from mpb200.problems import goal_mask
    make, kw, motion = _setup(mp, orc, name)
    P = make()
    mp.gmtstar(P, lam=1.0, edge_checks="lazy", **kw)                  # the roadmap, to pick free samples from
    N = len(P.V)
    free = np.flatnonzero(fx_bits(P.V.points_free(P.CC, P.SS), N))
    rng = np.random.Generator(np.random.PCG64(11))
    inits = [1] + [int(i) + 1 for i in rng.choice(free, 2, replace=False)]
    goals = [P.goal] + [mp.StateGoal(P.V.V[int(j)]) for j in rng.choice(free, 2, replace=False)]
    lams = [1.0, 0.25, 4.0]
    P.V.close()
    P = make()
    sols = mp.gmtstar_batch(P, inits, goals, lam=lams, edge_checks="lazy", **kw)
    F_tab, B_tab = _fetch_tables(P.V, kw)
    V, SS = P.V.V, P.SS
    col = lambda T, v: (T.rowval[T.colptr[v - 1] - 1:T.colptr[v] - 1], T.nzval[T.colptr[v - 1] - 1:T.colptr[v] - 1])
    F = fx_bits(P.V.points_free(P.CC, SS), N)
    inb = np.all((SS.lo <= V) & (V <= SS.hi), axis=1)
    check = motion(P)
    for q, sol in enumerate(sols):
        m = sol.metadata
        ref = gmt_oracle(N, goal_mask(V, goals[q], SS), lambda v: col(F_tab, v), lambda v: col(B_tab, v),
                         lambda i: bool(F[i]), lambda y0, x0: check(V[y0], V[x0]),
                         np.float64(lams[q]) * np.float64(m["r"]), init=inits[q], in_bounds=lambda y0: bool(inb[y0]))
        assert sol.status == ("solved" if ref["solved"] else "failed"), q
        assert m["path"] == ref["path"] and np.array_equal(m["tree"], ref["tree"]), q
        assert m["costs"].tobytes() == ref["costs"].tobytes() and sol.cost == ref["cost"], q
        assert (m["iterations"], m["expansions"], m["checks"], m["checks_in_bounds"], m["segment_checks"]) == (
            ref["iterations"], ref["expansions"], ref["checks"], ref["checks_in_bounds"], ref["seg_checks"]), q
    assert sols[0].status == "solved"
    P.V.close()


@pytest.mark.parametrize("mode", ["table", "lazy"])
def test_outputs_do_not_depend_on_the_rest_of_the_batch(gpu, orc, mode):
    mp = gpu
    R = Roadmap(mp, orc, "2d_20k", mode)
    qs = R.queries
    rc, base, _ = R.batch(qs)
    assert rc == 0
    perm = np.random.Generator(np.random.PCG64(3)).permutation(len(qs))
    rc, outs, _ = R.batch([qs[i] for i in perm])
    assert rc == 0 and [outs[k] for k in np.argsort(perm)] == base
    sub = [1, 4, 7]
    rc, outs, _ = R.batch([qs[i] for i in sub])
    assert rc == 0 and outs == [base[i] for i in sub]
    rng = np.random.Generator(np.random.PCG64(99))
    extra = [(int(a) + 1, np.arange(R.N) == int(b), float(l)) for a, b, l in
             zip(rng.integers(1, R.N, 5), rng.integers(0, R.N, 5), (0.5, 2.0, 0.0, 1.0, 8.0))]
    mixed = extra[:2] + qs[:5] + extra[2:] + qs[5:]
    rc, outs, _ = R.batch(mixed)
    assert rc == 0 and outs[2:7] + outs[10:] == base
    R.close()


def _batch_outputs(mp, orc, name, mode):
    R = Roadmap(mp, orc, name, mode)
    rc, outs, res = R.batch(R.queries)
    assert rc == 0, R.lib.mpb200_last_error()
    R.close()
    return outs, res[0].grid_blocks


@pytest.mark.parametrize("mode", ["table", "lazy"])
def test_batch_is_deterministic_and_one_launch(gpu, orc, mode, tmp_path):
    mp = gpu
    name = "2d_20k" if mode == "table" else "reedsshepp"
    a, blocks = _batch_outputs(mp, orc, name, mode)
    b, _ = _batch_outputs(mp, orc, name, mode)
    assert a == b
    dump = str(tmp_path / "gmt_batch_child.npy")
    code = ("import sys, pickle; sys.path[:0] = [%r, %r]; import mpb200 as mp; mp.init(0)\n"
            "from oracle import oracle as orc; orc.lib()\n"
            "import test_gpu_gmt_batch as t\n"
            "o = t._batch_outputs(mp, orc, %r, %r)\n"
            "pickle.dump(o, open(%r, 'wb'))\n" % (ROOT, os.path.join(ROOT, "tests"), name, mode, dump))
    subprocess.run([sys.executable, "-c", code], check=True, env=dict(os.environ, MPB200_GMT_GRID="37"), cwd=ROOT)
    import pickle
    with open(dump, "rb") as f:
        c, blocks37 = pickle.load(f)
    assert blocks37 == 37 != blocks and c == a
    R = Roadmap(mp, orc, name, mode)
    before = R.lib.mpb200_launch_count()
    rc, _, _ = R.batch(R.queries)
    assert rc == 0 and R.lib.mpb200_launch_count() - before == 1
    R.close()


def test_batch_argument_checks(gpu, orc):
    mp = gpu
    from mpb200 import _lib
    R = Roadmap(mp, orc, "2d_2k", "table")
    qs = R.queries[:4]
    lib, NN = R.lib, R.NN
    ok = lambda: R.batch(qs)[0]
    other = mp.MetricNN(NN.V.copy())                                                 # a table of another sample set
    other.build_table_checked(0.05, R.P.CC, R.P.SS)
    launches = lib.mpb200_launch_count()

    def rejects(code, ds=None, nq=None, res=True, paths=True, cap=None, edges=None):
        ds = R.descs(qs) if ds is None else ds
        n = len(qs) if nq is None else nq
        rs = (_lib.GmtResult * max(n, 1))() if res else None
        cap = R.N if cap is None else cap
        p = np.empty((max(n, 1), max(cap, 1)), dtype=np.int64) if paths else None
        rc = lib.mpb200_gmt_plan_batch(NN.handle(), ds, n, edges, rs, None, _lib.ptr(p), cap, None, None)
        return rc == code

    assert rejects(EARG, nq=0) and rejects(EARG, nq=-3)
    assert lib.mpb200_gmt_plan_batch(NN.handle(), None, 2, None, (_lib.GmtResult * 2)(), None, None, 0, None,
                                     None) == EARG                                   # NULL descs
    assert rejects(EARG, res=False)                                                  # NULL res
    assert rejects(EARG, paths=False)                                                # NULL paths, path_cap > 0
    assert rejects(EARG, cap=-1)
    for field, bad in (("init", 0), ("init", R.N + 1), ("width", -1.0), ("width", float("nan")), ("goal_bits", None)):
        ds = R.descs(qs)
        setattr(ds[2], field, bad)                                                   # one bad query among good ones
        assert rejects(EARG, ds=ds), field
    for field, value in (("fwd", other.table.h), ("bwd", other.table.h), ("checkpts", 0),
                         ("space", ctypes.pointer(mp.UnitHypercube(2).desc()))):
        ds = R.descs(qs)
        setattr(ds[3], field, value)                                                 # shared fields that differ
        assert rejects(EARG, ds=ds), field
        ds = R.descs(qs)
        for i in range(len(qs)):
            setattr(ds[i], field, value)
        if field in ("fwd", "bwd"):
            assert rejects(EARG, ds=ds), field                                       # all alike, but of another set
    assert rejects(EARG, edges=ctypes.byref(_lib.GmtEdges(7, R.P.CC.handle(), None, 0.0, 0, 0.0, 0.0)))
    import torch
    total = torch.cuda.get_device_properties(0).total_memory
    nq = total // (52 * R.N) + 1                                                     # scratch > device memory
    one = R.descs(qs[:1])[0]
    ds = (_lib.GmtDesc * nq)(*([one] * nq))
    rs = (_lib.GmtResult * nq)()
    assert lib.mpb200_gmt_plan_batch(NN.handle(), ds, nq, None, rs, None, None, 0, None, None) == ENOMEM
    assert lib.mpb200_launch_count() == launches                                     # no rejection launched
    assert ok() == 0 and lib.mpb200_launch_count() == launches + 1
    other.close()
    R.close()


def test_batch_full_size_c2_equals_single_plans(gpu):
    """C2 (ISRR_2H, N = 1M, r from fmt_radius), lambda = 1, table mode: 16 queries"""
    mp = gpu
    from mpb200.problems import goal_mask
    N = 1_000_000
    SS = mp.UnitHypercube(2)
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    P = mp.MPProblem(SS, [0.1, 0.1], mp.BallGoal([0.9, 0.9], 0.01), CC)
    st, _, _ = mp.gmtstar(P, N, lam=1.0, seed=20240602)
    assert st == "solved"
    R = Roadmap.__new__(Roadmap)
    R.P, R.NN, R.N, R.r = P, P.V, N, P.solution.metadata["r"]
    R.DF = R.DB = P.V.table
    R.edges = None
    from mpb200 import _lib
    R.lib = _lib.lib()
    free = np.flatnonzero(fx_bits(P.V.points_free(CC, SS), N))
    rng = np.random.Generator(np.random.PCG64(2024))
    R.queries = [(int(a) + 1, goal_mask(P.V.V, mp.BallGoal(P.V.V[int(b)], 0.01), SS), 1.0)
                 for a, b in zip(rng.choice(free, 16), rng.choice(free, 16))]
    rc, outs, _ = R.batch(R.queries)
    assert rc == 0 and sum(o[0] for o in outs) > 0
    for i, q in enumerate(R.queries):
        rc1, one, _ = R.single(q)
        assert rc1 == 0 and outs[i] == one, i
    R.close()
