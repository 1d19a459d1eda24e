"""GMT* on the device (mpb200_gmt_plan through planners.gmtstar): at lambda = 0 it is fmtstar(edge_checks="table");
at lambda > 0 it equals the CPU restatement tests/oracle_gmt.py over the same tables and bits; outputs do not depend on
run or launch geometry; one launch per plan; and the argument checks of the C ABI."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import fixtures as fx
from oracle_gmt import gmt_oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BOXES6D = [np.array([[0.45, 0.55], [0.0, 0.6]] + [[0.0, 1.0]] * 4)]   # a wall across x1 = 0.5, open where x2 > 0.6


def _free_samples(orc, O, So, lo, hi, N, seed, init, goal):
    rng = np.random.Generator(np.random.PCG64(seed))
    lo, hi = np.asarray(lo, dtype=float), np.asarray(hi, dtype=float)
    cand = lo + rng.random((4 * N, len(lo))) * (hi - lo)
    cand = cand[orc.states_free(O, So, cand)][:N - 2]
    assert len(cand) == N - 2
    return np.vstack([init, cand, goal])


def _case(mp, orc, name):
    """-> (make: () -> MPProblem, planner kwargs)"""
    if name.startswith("2d"):
        N = {"2d_2k": 2000, "2d_20k": 20000, "2d_knn": 2000}[name]
        O, So = orc.Obstacles2D(fx.ISRR_2H), orc.StateSpace([0, 0], [1, 1])
        V = _free_samples(orc, O, So, [0, 0], [1, 1], N, 20240601, [0.1, 0.1], [0.9, 0.9])
        SS = mp.UnitHypercube(2)
        CC = mp.PointRobot2D(fx.product_shape(mp, fx.ISRR_2H))
        make = lambda: mp.MPProblem(SS, V[0], mp.PointGoal(V[-1]), CC, V=mp.MetricNN(V, SS.dist, V[0]))
        return make, (dict(connections="K") if name == "2d_knn" else {})
    if name in ("3d_boxes", "6d_boxes"):
        d = 3 if name == "3d_boxes" else 6
        boxes = fx.BOXES3D if d == 3 else BOXES6D
        O, So = orc.Boxes(boxes), orc.StateSpace([0] * d, [1] * d)
        V = _free_samples(orc, O, So, [0] * d, [1] * d, 3000, 7 + d, [0.1] * d, [0.9] * d)
        SS = mp.UnitHypercube(d)
        CC = mp.PointRobotNDBoxes([mp.BoxBounds(b) for b in boxes])
        make = lambda: mp.MPProblem(SS, V[0], mp.PointGoal(V[-1]), CC, V=mp.MetricNN(V, SS.dist, V[0]))
        return make, dict(rm=1.5 if d == 3 else 1.2)
    if name == "double_integrator":
        SS = mp.DoubleIntegrator(2, vmax=0.5)
        O = orc.Boxes(fx.BOXES2D)
        So = orc.StateSpace(SS.lo, SS.hi, ("matrix", np.hstack([np.eye(2), np.zeros((2, 2))])))
        V = _free_samples(orc, O, So, SS.lo, SS.hi, 1200, 20240604, [0.1, 0.1, 0, 0], [0.9, 0.9, 0, 0])
        CC = mp.PointRobotNDBoxes([mp.BoxBounds(b) for b in fx.BOXES2D])
        make = lambda: mp.MPProblem(SS, V[0], mp.StateGoal(V[-1]), CC, V=mp.QuasiMetricNN(V, SS.dist, V[0]))
        return make, dict(r=1.0)
    kind = name
    SS = (mp.ReedsSheppMetricSpace if kind == "reedsshepp" else mp.DubinsQuasiMetricSpace)(0.05, 1.0)
    O = orc.Boxes(fx.BOXES2D)
    So = orc.StateSpace(SS.lo, SS.hi, ("view", [1, 2]))
    V = _free_samples(orc, O, So, SS.lo, SS.hi, 1500, 15, [0.1, 0.1, 0.0], [0.9, 0.9, 0.0])
    CC = mp.PointRobotNDBoxes([mp.BoxBounds(b) for b in fx.BOXES2D])
    NNcls = mp.MetricNN if kind == "reedsshepp" else mp.QuasiMetricNN
    make = lambda: mp.MPProblem(SS, V[0], mp.StateGoal(V[-1]), CC, V=NNcls(V, SS.dist, V[0]))
    return make, dict(r=0.25)


CASES = ["2d_2k", "2d_20k", "3d_boxes", "6d_boxes", "double_integrator", "reedsshepp", "dubins", "2d_knn"]


@pytest.mark.parametrize("name", CASES)
def test_gmt_at_lambda_zero_is_fmtstar(gpu, orc, name):
    mp = gpu
    make, kw = _case(mp, orc, name)
    Pf, Pg = make(), make()
    st_f, cost_f, _ = mp.fmtstar(Pf, edge_checks="table", **kw)
    st_g, cost_g, _ = mp.gmtstar(Pg, lam=0.0, **kw)
    mf, mg = Pf.solution.metadata, Pg.solution.metadata
    assert st_f == st_g == "solved"
    assert mg["path"] == mf["path"] and np.array_equal(mg["tree"], mf["tree"])
    assert np.float64(cost_g).tobytes() == np.float64(cost_f).tobytes()
    assert mg["collision_checks"] == mf["collision_checks"] > 0
    assert mg["precomputed_edge_checks"] == mf["precomputed_edge_checks"]
    assert mg["iterations"] == mg["expansions"] and mg["planner"] == "GMTstar"
    Pf.V.close(); Pg.V.close()


def _tables_of(NN, name, kw):
    """the device tables gmtstar planned over, fetched: (DF, DB, DB edge bits)"""
    from mpb200 import _lib
    if kw.get("connections") == "K":
        DF, DB = (NN.table_mknn, NN.table_knn) if hasattr(NN, "table_knn") else (NN.table_mknnF, NN.table_knnB)
    elif hasattr(NN, "tableF"):
        DF, DB = NN.tableF, NN.tableB
    else:
        DF = DB = NN.table
    f, b = NN.fetch_table(DF, "gF"), NN.fetch_table(DB, "gB")
    bits = np.empty((DB.nnz + 63) // 64, dtype=np.uint64)
    _lib.check(_lib.lib().mpb200_table_fetch_edge_bits(DB.h, _lib.ptr(bits)))
    return f, b, fx_bits(bits, DB.nnz)


def fx_bits(chunks, n):
    return np.unpackbits(np.ascontiguousarray(chunks).view(np.uint8), bitorder="little")[:n].astype(bool)


def _oracle_over(P, F_tab, B_tab, ebits, lam, checkpts=True):
    V, N = P.V.V, len(P.V)
    SS = P.SS
    col = lambda T, v: (T.rowval[T.colptr[v - 1] - 1:T.colptr[v] - 1], T.nzval[T.colptr[v - 1] - 1:T.colptr[v] - 1])

    def edge(y0, x0):
        lo, hi = B_tab.colptr[x0] - 1, B_tab.colptr[x0 + 1] - 1
        e = lo + int(np.flatnonzero(B_tab.rowval[lo:hi] == y0 + 1)[0])
        return bool(ebits[e]), 1

    F = fx_bits(P.V.points_free(P.CC, SS), N)
    from mpb200.problems import goal_mask
    inb = np.all((SS.lo <= V) & (V <= SS.hi), axis=1)
    return gmt_oracle(N, goal_mask(V, P.goal, SS), lambda v: col(F_tab, v), lambda v: col(B_tab, v),
                      lambda i: bool(F[i]), edge, np.float64(lam) * np.float64(P.solution.metadata["r"]),
                      checkpts=checkpts, in_bounds=lambda y0: bool(inb[y0]))


@pytest.mark.parametrize("name", CASES)
def test_gmt_at_positive_lambda_equals_the_cpu_restatement(gpu, orc, name):
    mp = gpu
    make, kw = _case(mp, orc, name)
    P = make()
    for lam in (0.25, 1.0, 4.0):
        st, cost, _ = mp.gmtstar(P, lam=lam, **kw)
        m = P.solution.metadata
        F_tab, B_tab, ebits = _tables_of(P.V, name, kw)
        ref = _oracle_over(P, F_tab, B_tab, ebits, lam)
        assert ref["solved"] and st == "solved", lam
        assert m["path"] == ref["path"] and np.array_equal(m["tree"], ref["tree"]), lam
        assert m["costs"].tobytes() == ref["costs"].tobytes() and cost == ref["cost"], lam
        assert (m["iterations"], m["expansions"]) == (ref["iterations"], ref["expansions"]), lam
        assert (m["checks"], m["checks_in_bounds"]) == (ref["checks"], ref["checks_in_bounds"]), lam
    P.V.close()


def _plan_outputs(mp, make, kw, lam):
    P = make()
    mp.gmtstar(P, lam=lam, **kw)
    m = P.solution.metadata
    out = (m["tree"].tobytes(), m["costs"].tobytes(), tuple(m["path"]), np.float64(m["cost"]).tobytes(),
           m["iterations"], m["expansions"], m["checks"], m["checks_in_bounds"])
    P.V.close()
    return out, m["grid_blocks"]


def test_gmt_is_deterministic_across_runs_and_grid_sizes(gpu, orc, tmp_path):
    mp = gpu
    make, kw = _case(mp, orc, "2d_20k")
    a, blocks = _plan_outputs(mp, make, kw, 1.0)
    b, _ = _plan_outputs(mp, make, kw, 1.0)
    assert a == b
    dump = str(tmp_path / "gmt_child.npz")
    code = ("import sys, numpy as np; sys.path[:0] = [%r, %r]; import mpb200 as mp; mp.init(0)\n"
            "from oracle import oracle as orc; orc.lib()\n"
            "import test_gpu_gmt as t\n"
            "make, kw = t._case(mp, orc, '2d_20k')\n"
            "o, blocks = t._plan_outputs(mp, make, kw, 1.0)\n"
            "np.savez(%r, blocks=blocks, **{'o%%d' %% i: np.frombuffer(x, np.uint8) if isinstance(x, bytes) else np.asarray(x) for i, x in enumerate(o)})\n"
            % (ROOT, os.path.join(ROOT, "tests"), dump))
    env = dict(os.environ, MPB200_GMT_GRID="37")
    subprocess.run([sys.executable, "-c", code], check=True, env=env, cwd=ROOT)
    with np.load(dump) as z:
        assert int(z["blocks"]) == 37 != blocks
        for i, x in enumerate(a):
            got = z["o%d" % i]
            assert (got.tobytes() == x) if isinstance(x, bytes) else np.array_equal(got, np.asarray(x)), i


def test_gmt_launches_once_per_plan(gpu, orc):
    mp = gpu
    lib = mp.load()
    make, kw = _case(mp, orc, "2d_2k")
    P = make()
    counts = []
    for lam in (0.0, 1.0, 8.0):
        mp.gmtstar(P, lam=lam, **kw)                      # tables first (their launches are not the planner's)
        before = lib.mpb200_launch_count()
        _replan(mp, P, lam)
        counts.append((lib.mpb200_launch_count() - before, P.solution.metadata["iterations"]))
    assert len({it for _, it in counts}) == 3             # very different iteration counts ...
    assert {n for n, _ in counts} == {1}                  # ... one kernel launch each
    P.V.close()


def _gmt_call(mp, NN, DF, DB, goal_mask_bool, init=1, width=0.0, checkpts=1, space=None, path_cap=None, tree=True):
    from mpb200 import _lib
    N = len(NN)
    chunks = np.zeros((N + 63) // 64 * 8, dtype=np.uint8)
    pk = np.packbits(goal_mask_bool, bitorder="little")
    chunks[:len(pk)] = pk
    chunks = chunks.view(np.uint64)
    desc = _lib.GmtDesc(DF.h if DF is not None else None, DB.h if DB is not None else None, _lib.ptr(chunks), init,
                        width, checkpts, ctypes.pointer(space) if space is not None else None)
    res = _lib.GmtResult()
    cap = N if path_cap is None else path_cap
    path = np.full(max(cap, 1), -7, dtype=np.int64)
    t = np.empty(N, dtype=np.int64) if tree else None
    rc = _lib.lib().mpb200_gmt_plan(NN.handle(), ctypes.byref(desc), ctypes.byref(res), _lib.ptr(path), cap,
                                    _lib.ptr(t), None)
    return rc, res, path


def _replan(mp, P, lam):
    """plan again over the tables gmtstar left on the device (no rebuild)"""
    from mpb200.problems import goal_mask
    NN = P.V
    rc, res, _ = _gmt_call(mp, NN, NN.table, NN.table, goal_mask(NN.V, P.goal, P.SS),
                           width=lam * P.solution.metadata["r"])
    assert rc == 0
    P.solution.metadata["iterations"] = res.iterations


def test_gmt_edge_cases(gpu, orc):
    mp = gpu
    SS = mp.UnitHypercube(2)
    CC = mp.PointRobotNDBoxes([mp.BoxBounds(b) for b in fx.BOXES2D])
    # init in collision: failed, as fmtstar
    P = mp.MPProblem(SS, [0.08, 0.43], mp.PointGoal([0.9, 0.9]), CC)
    assert mp.gmtstar(P, 100) == float("inf") and P.status == "failed"
    make, kw = _case(mp, orc, "2d_2k")
    # init is a goal: 0 iterations, cost 0
    P = make()
    P.goal = mp.PointGoal(P.V.V[0])
    st, cost, _ = mp.gmtstar(P, lam=1.0)
    m = P.solution.metadata
    assert st == "solved" and cost == 0.0 and m["path"] == [1] and m["iterations"] == 0 and m["checks"] == 0
    # an unreachable goal (a point inside an obstacle is never a free sample): failed, cost inf
    P2 = make()
    P2.goal = mp.PointGoal([0.1, 0.45])
    st, cost, _ = mp.gmtstar(P2, lam=1.0)
    assert st == "failed" and cost == float("inf") and P2.solution.metadata["path"] == []
    assert P2.solution.metadata["iterations"] > 0
    # checkpts=False equals the oracle with every sample free
    P3 = make()
    st, cost, _ = mp.gmtstar(P3, lam=1.0, checkpts=False)
    F_tab, B_tab, ebits = _tables_of(P3.V, "2d_2k", {})
    ref = _oracle_over(P3, F_tab, B_tab, ebits, 1.0, checkpts=False)
    assert st == "solved" and P3.solution.metadata["path"] == ref["path"]
    assert P3.solution.metadata["costs"].tobytes() == ref["costs"].tobytes()
    # N = 1: init alone, not a goal -> failed after one iteration; a goal -> solved
    V1 = np.array([[0.1, 0.1]])
    NN1 = mp.MetricNN(V1)
    NN1.build_table_checked(0.1, CC, SS)
    NN1.points_free(CC, SS, fetch=False)
    rc, res, _ = _gmt_call(mp, NN1, NN1.table, NN1.table, np.array([False]))
    assert rc == 0 and not res.solved and res.iterations == 1 and res.path_len == 0 and res.cost == float("inf")
    rc, res, path = _gmt_call(mp, NN1, NN1.table, NN1.table, np.array([True]))
    assert rc == 0 and res.solved and res.path_len == 1 and path[0] == 1
    NN1.close()
    # path_cap too small: path_len reported, nothing written
    NN = P3.V
    goal = np.all(NN.V == NN.V[-1], axis=1)
    rc, res, path = _gmt_call(mp, NN, NN.table, NN.table, goal, width=0.01)
    assert rc == 0 and res.solved and res.path_len > 2 and path[0] == 1
    rc, res2, path = _gmt_call(mp, NN, NN.table, NN.table, goal, width=0.01, path_cap=res.path_len - 1)
    assert rc == 0 and res2.path_len == res.path_len and np.all(path == -7)
    # MPB200_EARG cases
    EARG = -1
    other = mp.MetricNN(NN.V.copy())                                   # same N and d, another sample set
    other.build_table_checked(0.05, CC, SS)
    assert _gmt_call(mp, NN, other.table, NN.table, goal)[0] == EARG
    assert _gmt_call(mp, NN, NN.table, other.table, goal)[0] == EARG
    other.close()
    assert _gmt_call(mp, NN, NN.table, NN.table, goal, init=0)[0] == EARG
    assert _gmt_call(mp, NN, NN.table, NN.table, goal, width=-1.0)[0] == EARG
    assert _gmt_call(mp, NN, NN.table, NN.table, goal, width=float("nan"))[0] == EARG
    NN.build_table(0.05)                                                # new contents, no edge bits yet
    assert _gmt_call(mp, NN, NN.table, NN.table, goal)[0] == EARG
    NN.edges_free(NN.table, CC, SS, fetch=False)
    assert _gmt_call(mp, NN, NN.table, NN.table, goal)[0] == 0
    fresh = mp.MetricNN(NN.V.copy())                                    # no point bits yet
    fresh.build_table_checked(0.05, CC, SS)
    assert _gmt_call(mp, fresh, fresh.table, fresh.table, goal)[0] == EARG
    assert _gmt_call(mp, fresh, fresh.table, fresh.table, goal, checkpts=0)[0] == 0
    fresh.set_query_range(0, 1000)                                      # point bits of a shard only
    fresh.points_free(CC, SS, fetch=False)
    assert _gmt_call(mp, fresh, fresh.table, fresh.table, goal)[0] == EARG
    fresh.build_table_checked(0.05, CC, SS)                             # a sharded table
    assert _gmt_call(mp, fresh, fresh.table, fresh.table, goal, checkpts=0)[0] == EARG
    fresh.close()
    P3.V.close(); P.V.close(); P2.V.close()


def test_gmt_full_size_c2_matches_a_vectorised_restatement(gpu):
    """C2 (ISRR_2H, N = 1M, r from fmt_radius), lambda = 1, against a numpy restatement over the fetched tables"""
    mp = gpu
    N = 1_000_000
    SS = mp.UnitHypercube(2)
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    P = mp.MPProblem(SS, [0.1, 0.1], mp.BallGoal([0.9, 0.9], 0.01), CC)
    st, cost, _ = mp.gmtstar(P, N, lam=1.0, seed=20240602)
    m = P.solution.metadata
    NN = P.V
    T = NN.fetch_table(NN.table)
    from mpb200 import _lib
    bits = np.empty((T.nnz + 63) // 64, dtype=np.uint64)
    _lib.check(_lib.lib().mpb200_table_fetch_edge_bits(NN.table.h, _lib.ptr(bits)))
    ref = _numpy_gmt(NN.V, T, fx_bits(bits, T.nnz), fx_bits(NN.points_free(CC, SS), N),
                     mp.problems.goal_mask(NN.V, P.goal, SS), np.float64(m["r"]) * np.float64(1.0))
    assert st == "solved" and ref["solved"]
    assert m["costs"].tobytes() == ref["costs"].tobytes() and np.array_equal(m["tree"], ref["tree"])
    assert m["path"] == ref["path"] and (m["iterations"], m["expansions"], m["checks"]) == (
        ref["iterations"], ref["expansions"], ref["checks"])
    NN.close()


def _numpy_gmt(V, T, ebits, F, goal, w):
    """the specification vectorised over whole iterations (symmetric r-ball table: DF = DB = T)"""
    N = len(V)
    cp, rv, nz = np.asarray(T.colptr) - 1, np.asarray(T.rowval) - 1, np.asarray(T.nzval)
    col_of = np.repeat(np.arange(N), np.diff(cp))
    C = np.zeros(N)
    A = np.zeros(N, dtype=np.int64)
    state = np.zeros(N, dtype=np.int8)          # 0 W, 1 H, 2 closed
    state[0] = 1
    it = exps = checks = 0
    while True:
        openv = np.flatnonzero(state == 1)
        if openv.size == 0:
            return dict(solved=False)
        thr = C[openv].min() + w
        G = openv[C[openv] <= thr]
        if goal[G].any():
            gs = G[goal[G]]
            g = gs[np.lexsort((gs, C[gs]))[0]]
            path = [int(g) + 1]
            while path[0] != 1:
                path.insert(0, int(A[path[0] - 1]))
            return dict(solved=True, costs=C, tree=A, path=path, iterations=it, expansions=exps, checks=checks)
        # candidates: rows of the columns of G that are unvisited and free
        sel = np.concatenate([np.arange(cp[g], cp[g + 1]) for g in G]) if G.size else np.zeros(0, np.int64)
        X = np.unique(rv[sel])
        X = X[(state[X] == 0) & F[X]]
        # entries of the columns of X whose row is open
        ent = np.concatenate([np.arange(cp[x], cp[x + 1]) for x in X]) if X.size else np.zeros(0, np.int64)
        ent = ent[state[rv[ent]] == 1]
        cost = C[rv[ent]] + nz[ent]
        order = np.lexsort((ent, cost, col_of[ent]))           # per column: cheapest, then first in storage
        ent, cost = ent[order], cost[order]
        first = np.ones(len(ent), dtype=bool)
        first[1:] = col_of[ent][1:] != col_of[ent][:-1]
        ent, cost = ent[first], cost[first]
        checks += len(ent)
        ok = ebits[ent]
        xs = col_of[ent][ok]
        C[xs], A[xs] = cost[ok], rv[ent][ok] + 1
        state[G] = 2
        state[xs] = 1
        it += 1
        exps += len(G)
