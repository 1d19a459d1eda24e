"""Lazy GMT* on the device (mpb200_gmt_plan_lazy through planners.gmtstar(edge_checks="lazy")): equal to table mode
on every problem kind and width; equal to tests/oracle_gmt.py run with the oracle's own per-pair motion checkers
(no device bits involved), segment count included; equal to fmtstar(edge_checks="lazy") at lambda = 0; blind to the
edge bits of the backward table; a replan on one roadmap against a new obstacle set; deterministic, one launch per
plan; the argument checks of the C ABI; C2 at full size."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import fixtures as fx
from oracle_gmt import gmt_oracle
from test_gpu_gmt import BOXES6D, CASES, _case, _free_samples, _gmt_call, fx_bits

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EARG = -1
LAMS = (0.0, 0.25, 1.0, 4.0)
EXTRA = ["lqg_di2_drift", "lqg_triple", "double_integrator_knn", "dubins_knn"]


def _lqg_case(mp, orc, name):
    import json
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "lq_general.json")))["systems"][name]
    A, B, c, R = (np.array(g[k]) for k in ("A", "B", "c", "R"))
    if name == "di2_drift":                                          # as tests/test_gpu_lq_general.py
        lo, hi = np.array([0, 0, -1.5, -1.5]), np.array([1, 1, 1.5, 1.5])
        C = np.hstack([np.eye(2), np.zeros((2, 2))])
        init, goal, N, r = [0.1, 0.1, 0, 0], [0.9, 0.9, 0, 0], 900, 1.0
    else:
        lo, hi = np.array([0, -1.0, -2.0]), np.array([1, 1.0, 2.0])
        C = np.array([[1.0, 0, 0], [0, 1.0, 0]])
        init, goal, N, r = [0.1, 0, 0], [0.9, 0, 0], 1500, 2.0          # init reaches 14 samples within r
    SS = mp.linearquadratic.LinearQuadraticQuasiMetricSpace(lo, hi, A, B, c, R, C)
    O, So = orc.Obstacles2D(fx.ISRR_2H), orc.StateSpace(lo, hi, ("matrix", C))
    V = _free_samples(orc, O, So, lo, hi, N, 20240605 + len(init), init, goal)
    CC = mp.PointRobot2D(fx.product_shape(mp, fx.ISRR_2H))
    make = lambda: mp.MPProblem(SS, V[0], mp.StateGoal(V[-1]), CC, V=mp.QuasiMetricNN(V, SS.dist, V[0]))
    L = orc.LinearQuadraticGeneral(A, B, c, R)
    return make, dict(r=r), lambda P: (lambda v, w: L.is_free_motion(O, So, P.V.r, v, w))


def _setup(mp, orc, name):
    """-> (make, planner kwargs, oracle motion check: P -> ((v, w) -> (free, segment tests)))"""
    if name.startswith("lqg_"):
        return _lqg_case(mp, orc, name[4:])
    knn = name.endswith("_knn") and name != "2d_knn"
    make, kw = _case(mp, orc, name[:-4] if knn else name)
    if knn:
        kw = dict(kw, connections="K")
    base = name[:-4] if knn else name
    if base.startswith("2d"):
        O, So = orc.Obstacles2D(fx.ISRR_2H), orc.StateSpace([0, 0], [1, 1])
    elif base in ("3d_boxes", "6d_boxes"):
        d = 3 if base == "3d_boxes" else 6
        O = orc.Boxes(fx.BOXES3D if d == 3 else BOXES6D)
        So = orc.StateSpace([0] * d, [1] * d)
    else:
        O = orc.Boxes(fx.BOXES2D)
    if base.startswith("2d") or base in ("3d_boxes", "6d_boxes"):
        def straight(P):
            return lambda v, w: (lambda ok, n: (bool(ok[0]), n))(*orc.motions_free_straight(O, So, v, w))
        return make, kw, straight
    if base == "double_integrator":
        def lq(P):
            SS = P.SS
            So = orc.StateSpace(SS.lo, SS.hi, ("matrix", np.hstack([np.eye(2), np.zeros((2, 2))])))
            L = orc.DoubleIntegratorLQ(2)
            return lambda v, w: L.is_free_motion(O, So, P.V.r, v, w)
        return make, kw, lq

    def car(P):
        m = P.V.dist.m
        So = orc.StateSpace(P.SS.lo, P.SS.hi, ("view", [1, 2]))
        C = orc.SimpleCar(m.kind, m.r, m.s)
        return lambda v, w: C.is_free_motion(O, So, v, w)
    return make, kw, car


def _outputs(P, cost):
    m = P.solution.metadata
    return (m["tree"].tobytes(), m["costs"].tobytes(), tuple(m["path"]), np.float64(cost).tobytes(), m["iterations"],
            m["expansions"], m["checks"], m["checks_in_bounds"], m["collision_checks"])


def _fetch_tables(NN, kw):
    """the device tables gmtstar planned over, without edge bits: (DF, DB) as host CSC"""
    if kw.get("connections") == "K":
        DF, DB = (NN.table_mknn, NN.table_knn) if hasattr(NN, "table_knn") else (NN.table_mknnF, NN.table_knnB)
    elif hasattr(NN, "tableF"):
        DF, DB = NN.tableF, NN.tableB
    else:
        DF = DB = NN.table
    return NN.fetch_table(DF, "gF"), NN.fetch_table(DB, "gB")


def _lazy_oracle(P, F_tab, B_tab, motion, w, F=None):
    """gmt_oracle over the fetched tables with the oracle's motion check; w = lambda * r"""
    V, N, SS = P.V.V, len(P.V), P.SS
    col = lambda T, v: (T.rowval[T.colptr[v - 1] - 1:T.colptr[v] - 1], T.nzval[T.colptr[v - 1] - 1:T.colptr[v] - 1])
    if F is None:
        F = fx_bits(P.V.points_free(P.CC, SS), N)
    from mpb200.problems import goal_mask
    inb = np.all((SS.lo <= V) & (V <= SS.hi), axis=1)
    return gmt_oracle(N, goal_mask(V, P.goal, SS), lambda v: col(F_tab, v), lambda v: col(B_tab, v),
                      lambda i: bool(F[i]), lambda y0, x0: motion(V[y0], V[x0]),
                      w, in_bounds=lambda y0: bool(inb[y0]))


@pytest.mark.parametrize("name", CASES + EXTRA)
def test_lazy_equals_table(gpu, orc, name):
    mp = gpu
    make, kw, _ = _setup(mp, orc, name)
    Pt, Pl = make(), make()
    for lam in LAMS:
        st_t, cost_t, _ = mp.gmtstar(Pt, lam=lam, **kw)
        st_l, cost_l, _ = mp.gmtstar(Pl, lam=lam, edge_checks="lazy", **kw)
        mt, ml = Pt.solution.metadata, Pl.solution.metadata
        assert st_t == st_l and _outputs(Pl, cost_l) == _outputs(Pt, cost_t), lam
        assert ml["edge_checks"] == "lazy" and ml["precomputed_edge_checks"] == 0 and mt["edge_checks"] == "table"
        assert "segment_checks" not in mt and 0 < ml["segment_checks"] < mt["precomputed_edge_checks"], lam
    Pt.V.close(); Pl.V.close()


@pytest.mark.parametrize("name", CASES + EXTRA[:2])
def test_lazy_equals_the_oracle_with_its_own_motion_checks(gpu, orc, name):
    mp = gpu
    make, kw, motion = _setup(mp, orc, name)
    P = make()
    for lam in (0.25, 1.0):
        st, cost, _ = mp.gmtstar(P, lam=lam, edge_checks="lazy", **kw)
        m = P.solution.metadata
        F_tab, B_tab = _fetch_tables(P.V, kw)
        ref = _lazy_oracle(P, F_tab, B_tab, motion(P), np.float64(lam) * np.float64(m["r"]))
        assert st == ("solved" if ref["solved"] else "failed"), lam
        assert m["path"] == ref["path"] and np.array_equal(m["tree"], ref["tree"]), lam
        assert m["costs"].tobytes() == ref["costs"].tobytes() and cost == ref["cost"], lam
        assert (m["iterations"], m["expansions"]) == (ref["iterations"], ref["expansions"]), lam
        assert (m["checks"], m["checks_in_bounds"]) == (ref["checks"], ref["checks_in_bounds"]), lam
        assert m["segment_checks"] == ref["seg_checks"] > 0, lam
        if name in ("2d_2k", "2d_20k", "2d_knn", "3d_boxes", "6d_boxes"):
            assert m["segment_checks"] == m["checks_in_bounds"]
    P.V.close()


@pytest.mark.parametrize("name", ["2d_2k", "3d_boxes", "double_integrator", "reedsshepp", "dubins"])
def test_lazy_at_lambda_zero_is_lazy_fmtstar(gpu, orc, name):
    mp = gpu
    make, kw = _case(mp, orc, name)
    Pf, Pg = make(), make()
    st_f, cost_f, _ = mp.fmtstar(Pf, edge_checks="lazy", **kw)
    st_g, cost_g, _ = mp.gmtstar(Pg, lam=0.0, edge_checks="lazy", **kw)
    mf, mg = Pf.solution.metadata, Pg.solution.metadata
    assert st_f == st_g == "solved"
    assert mg["path"] == mf["path"] and np.array_equal(mg["tree"], mf["tree"])
    assert np.float64(cost_g).tobytes() == np.float64(cost_f).tobytes()
    assert mg["collision_checks"] == mf["collision_checks"] > 0
    Pf.V.close(); Pg.V.close()


def _goal_chunks(mask):
    chunks = np.zeros((len(mask) + 63) // 64 * 8, dtype=np.uint8)
    pk = np.packbits(mask, bitorder="little")
    chunks[:len(pk)] = pk
    return chunks.view(np.uint64)


def _lazy_call(NN, DF, DB, goal, edges, width=0.0, init=1, checkpts=1, space=None, seg=True):
    """mpb200_gmt_plan_lazy over the given device tables -> (rc, result, path, tree, costs, segment checks)"""
    from mpb200 import _lib
    N = len(NN)
    chunks = _goal_chunks(goal)
    desc = _lib.GmtDesc(DF.h, DB.h, _lib.ptr(chunks), init, width, checkpts,
                        ctypes.pointer(space) if space is not None else None)
    res = _lib.GmtResult()
    path = np.full(N, -7, dtype=np.int64)
    tree, costs = np.empty(N, dtype=np.int64), np.empty(N)
    segs = _lib.c_i64(-1)
    rc = _lib.lib().mpb200_gmt_plan_lazy(NN.handle(), ctypes.byref(desc), ctypes.byref(edges) if edges else None,
                                         ctypes.byref(res), ctypes.byref(segs) if seg else None, _lib.ptr(path), N,
                                         _lib.ptr(tree), _lib.ptr(costs))
    return rc, res, path[:max(res.path_len, 0)], tree, costs, segs.value


def _straight(CC):
    from mpb200 import _lib
    return _lib.GmtEdges(_lib.GMT_EDGES_STRAIGHT, CC.handle(), None, 0.0, 0, 0.0, 0.0)


def _edge_bits(NN, t):
    from mpb200 import _lib
    bits = np.empty((t.nnz + 63) // 64, dtype=np.uint64)
    _lib.check(_lib.lib().mpb200_table_fetch_edge_bits(t.h, _lib.ptr(bits)))
    return bits


def test_lazy_ignores_the_edge_bits(gpu, orc):
    mp = gpu
    from mpb200.problems import goal_mask
    make, kw, motion = _setup(mp, orc, "2d_2k")
    P = make()
    st, cost, _ = mp.gmtstar(P, lam=1.0, edge_checks="lazy")      # a table that never had edge bits
    assert st == "solved"
    NN, SS, CC = P.V, P.SS, P.CC
    lazy0 = _outputs(P, cost)
    goal, w, space = goal_mask(NN.V, P.goal, SS), 1.0 * P.solution.metadata["r"], SS.desc()
    # bits computed for another obstacle set: ignored
    other = mp.PointRobot2D(fx.product_shape(mp, fx.TRI_BALLS))
    NN.edges_free(NN.table, other, SS, fetch=False)
    before = _edge_bits(NN, NN.table).copy()
    rc, res, path, tree, costs, segs = _lazy_call(NN, NN.table, NN.table, goal, _straight(CC), width=w, space=space)
    assert rc == 0 and np.array_equal(_edge_bits(NN, NN.table), before)
    assert list(path) == P.solution.metadata["path"] and tree.tobytes() == lazy0[0] and costs.tobytes() == lazy0[1]
    F_tab, B_tab = _fetch_tables(NN, {})
    ref = _lazy_oracle(P, F_tab, B_tab, motion(P), np.float64(w))
    assert list(path) == ref["path"] and costs.tobytes() == ref["costs"].tobytes() and segs == ref["seg_checks"]
    # table mode after the bits are recomputed for these obstacles gives the same plan
    NN.edges_free(NN.table, CC, SS, fetch=False)
    rc, rt, pt = _gmt_call(mp, NN, NN.table, NN.table, goal, width=w, space=space)
    assert rc == 0 and list(pt[:rt.path_len]) == list(path) and rt.cost == res.cost
    assert (rt.iterations, rt.expansions, rt.checks, rt.checks_in_bounds) == (
        res.iterations, res.expansions, res.checks, res.checks_in_bounds)
    other.close()
    NN.close()


def test_replan_on_one_roadmap_with_a_new_obstacle(gpu, orc):
    mp = gpu
    from mpb200 import _lib
    from mpb200.problems import goal_mask
    lib = _lib.lib()
    make, kw, _ = _setup(mp, orc, "2d_2k")
    P = make()
    NN, SS, CC = P.V, P.SS, P.CC
    NN.build_table(0.08)                                           # the roadmap: one table, no edge bits
    NN.points_free(CC, SS, fetch=False)
    goal, space = goal_mask(NN.V, P.goal, SS), SS.desc()
    So = orc.StateSpace([0, 0], [1, 1])
    F_tab, B_tab = _fetch_tables(NN, {})
    c0 = lib.mpb200_launch_count()
    rc, r1, path1, tree1, costs1, segs1 = _lazy_call(NN, NN.table, NN.table, goal, _straight(CC), width=0.08,
                                                     space=space)
    c1 = lib.mpb200_launch_count()
    assert rc == 0 and r1.solved and c1 - c0 == 1
    O1 = orc.Obstacles2D(fx.ISRR_2H)
    ref1 = _lazy_oracle(P, F_tab, B_tab, lambda v, w: (lambda ok, n: (bool(ok[0]), n))(
        *orc.motions_free_straight(O1, So, v, w)), 0.08, F=orc.states_free(O1, So, NN.V))
    assert list(path1) == ref1["path"] and costs1.tobytes() == ref1["costs"].tobytes() and segs1 == ref1["seg_checks"]
    # a blocker across the middle edge of the first solution
    k = len(path1) // 2
    centre = 0.5 * (NN.V[path1[k - 1] - 1] + NN.V[path1[k] - 1])
    CC2 = mp.addobstacle(CC, mp.Circle(centre, 0.02))
    spec2 = ("compound", [fx.ISRR_2H, ("circle", tuple(centre), 0.02)])
    O2 = orc.Obstacles2D(spec2)
    NN.points_free(CC2, SS, fetch=False)                           # the only launch between the plans
    c2 = lib.mpb200_launch_count()
    rc, r2, path2, tree2, costs2, segs2 = _lazy_call(NN, NN.table, NN.table, goal, _straight(CC2), width=0.08,
                                                     space=space)
    assert rc == 0 and lib.mpb200_launch_count() - c2 == 1
    ref2 = _lazy_oracle(P, F_tab, B_tab, lambda v, w: (lambda ok, n: (bool(ok[0]), n))(
        *orc.motions_free_straight(O2, So, v, w)), 0.08, F=orc.states_free(O2, So, NN.V))
    assert bool(r2.solved) == ref2["solved"] and list(path2) == ref2["path"]
    assert costs2.tobytes() == ref2["costs"].tobytes() and tree2.tobytes() == ref2["tree"].tobytes()
    assert segs2 == ref2["seg_checks"] and (r2.checks, r2.iterations) == (ref2["checks"], ref2["iterations"])
    assert list(path2) != list(path1)
    if r2.solved:
        seg_ok, _ = orc.motions_free_straight(O2, So, NN.V[path2[:-1] - 1], NN.V[path2[1:] - 1])
        assert seg_ok.all()
    assert NN.table.nnz == F_tab.nnz
    CC2.close()
    NN.close()


def _plan_outputs(mp, orc, name):
    make, kw, _ = _setup(mp, orc, name)
    P = make()
    st, cost, _ = mp.gmtstar(P, lam=1.0, edge_checks="lazy", **kw)
    out = _outputs(P, cost) + (P.solution.metadata["segment_checks"],)
    blocks = P.solution.metadata["grid_blocks"]
    P.V.close()
    return out, blocks


@pytest.mark.parametrize("name", ["2d_20k", "reedsshepp"])
def test_lazy_is_deterministic_and_one_launch(gpu, orc, name, tmp_path):
    mp = gpu
    a, blocks = _plan_outputs(mp, orc, name)
    b, _ = _plan_outputs(mp, orc, name)
    assert a == b
    dump = str(tmp_path / "gmt_lazy_child.npz")
    code = ("import sys, numpy as np; sys.path[:0] = [%r, %r]; import mpb200 as mp; mp.init(0)\n"
            "from oracle import oracle as orc; orc.lib()\n"
            "import test_gpu_gmt_lazy as t\n"
            "o, blocks = t._plan_outputs(mp, orc, %r)\n"
            "np.savez(%r, blocks=blocks, **{'o%%d' %% i: np.frombuffer(x, np.uint8) if isinstance(x, bytes) else np.asarray(x) for i, x in enumerate(o)})\n"
            % (ROOT, os.path.join(ROOT, "tests"), name, dump))
    subprocess.run([sys.executable, "-c", code], check=True, env=dict(os.environ, MPB200_GMT_GRID="37"), cwd=ROOT)
    with np.load(dump) as z:
        assert int(z["blocks"]) == 37 != blocks
        for i, x in enumerate(a):
            got = z["o%d" % i]
            assert (got.tobytes() == x) if isinstance(x, bytes) else np.array_equal(got, np.asarray(x)), i
    # one launch per plan, over the tables the last gmtstar left
    from mpb200 import _lib
    from mpb200.problems import goal_mask
    lib = _lib.lib()
    make, kw, _ = _setup(mp, orc, name)
    P = make()
    mp.gmtstar(P, lam=1.0, edge_checks="lazy", **kw)
    NN = P.V
    DF, DB = (NN.table, NN.table) if hasattr(NN, "table") else (NN.tableF, NN.tableB)
    if name == "reedsshepp":
        m = NN.dist.m
        edges = _lib.GmtEdges(_lib.GMT_EDGES_CAR, P.CC.handle(), None, 0.0, m.kind, m.r, m.s)
    else:
        edges = _straight(P.CC)
    before = lib.mpb200_launch_count()
    rc, res, path, _, _, _ = _lazy_call(NN, DF, DB, goal_mask(NN.V, P.goal, P.SS), edges,
                                        width=P.solution.metadata["r"], space=P.SS.desc())
    assert rc == 0 and lib.mpb200_launch_count() - before == 1 and list(path) == P.solution.metadata["path"]
    NN.close()


def test_lazy_argument_checks(gpu, orc):
    mp = gpu
    from mpb200 import _lib
    from mpb200.problems import goal_mask
    make, kw, _ = _setup(mp, orc, "2d_2k")
    P = make()
    mp.gmtstar(P, lam=1.0, edge_checks="lazy")
    NN, SS, CC = P.V, P.SS, P.CC
    goal, sp = goal_mask(NN.V, P.goal, SS), SS.desc()
    call = lambda edges, **k: _lazy_call(NN, NN.table, NN.table, goal, edges, **dict(dict(space=sp), **k))[0]
    E = lambda kind=_lib.GMT_EDGES_STRAIGHT, obs=CC.handle(), lq=None, r=0.0, ck=0, tr=0.0, s=0.0: _lib.GmtEdges(
        kind, obs, lq, r, ck, tr, s)
    assert call(E()) == 0 and call(E(), seg=False) == 0
    assert call(None) == EARG                                          # NULL edges
    assert call(E(obs=None)) == EARG                                   # NULL obstacles
    assert call(E(kind=7)) == EARG                                     # unknown kind
    assert call(E(), space=None) == EARG                               # no space
    assert call(E(), space=mp.UnitHypercube(3).desc()) == EARG         # space->n != d
    assert call(E(), init=0) == EARG and call(E(), width=-1.0) == EARG and call(E(), width=float("nan")) == EARG
    assert call(E(kind=_lib.GMT_EDGES_CAR, ck=0, tr=0.05, s=1.0)) == EARG      # car kind with d = 2
    assert call(E(kind=_lib.GMT_EDGES_LQ, r=1.0)) == EARG                      # LQ without a system
    DI = mp.DoubleIntegrator(2)
    assert call(E(kind=_lib.GMT_EDGES_LQ, lq=DI.dist.handle(), r=1.0)) == EARG  # 4 states != d = 2
    DI1 = mp.DoubleIntegrator(1)                                                # 2 states: d matches
    for r in (0.0, -1.0, float("nan"), float("inf")):
        assert call(E(kind=_lib.GMT_EDGES_LQ, lq=DI1.dist.handle(), r=r)) == EARG, r
    boxes3 = mp.PointRobotNDBoxes([mp.BoxBounds(b) for b in fx.BOXES3D])
    assert call(E(obs=boxes3.handle())) == EARG                        # 3-D boxes in a 2-D workspace
    NN.build_table(0.05)                                               # new contents: no edge bits, still fine
    assert call(E()) == 0
    # car kinds on SE2 samples
    make3, kw3, _ = _setup(mp, orc, "reedsshepp")
    P3 = make3()
    mp.gmtstar(P3, lam=1.0, edge_checks="lazy", **kw3)
    N3, m = P3.V, P3.V.dist.m
    call3 = lambda edges, **k: _lazy_call(N3, N3.table, N3.table, goal_mask(N3.V, P3.goal, P3.SS), edges,
                                          **dict(dict(space=P3.SS.desc()), **k))[0]
    car = lambda ck=m.kind, tr=m.r, s=m.s, obs=P3.CC.handle(): E(kind=_lib.GMT_EDGES_CAR, obs=obs, ck=ck, tr=tr, s=s)
    assert call3(car()) == 0
    assert call3(car(ck=5)) == EARG
    for bad in (0.0, -0.1, float("nan"), float("inf")):
        assert call3(car(tr=bad)) == EARG and call3(car(s=bad)) == EARG, bad
    assert call3(car(obs=boxes3.handle())) == EARG                     # box dimension 3 != workspace dimension 2
    sd3 = mp.UnitHypercube(3).desc()                                   # identity view: 3-D workspace, 2-D compound
    assert call3(car(obs=mp.PointRobot2D(fx.product_shape(mp, fx.ISRR_2H)).handle()), space=sd3) == EARG
    boxes3.close()
    N3.close(); NN.close()


def test_lazy_full_size_c2_equals_table(gpu):
    mp = gpu
    N = 1_000_000
    runs = []
    for mode in ("table", "lazy"):
        SS = mp.UnitHypercube(2)
        CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
        P = mp.MPProblem(SS, [0.1, 0.1], mp.BallGoal([0.9, 0.9], 0.01), CC)
        st, cost, _ = mp.gmtstar(P, N, lam=1.0, seed=20240602, edge_checks=mode)
        m = P.solution.metadata
        runs.append((st, m["tree"].tobytes(), m["costs"].tobytes(), m["path"], m["checks"], m["checks_in_bounds"],
                     m.get("segment_checks")))
        P.V.close()
    assert runs[0][0] == "solved" and runs[0][:6] == runs[1][:6]
    assert runs[1][6] == runs[1][5] > 0
