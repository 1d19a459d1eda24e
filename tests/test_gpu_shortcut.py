"""Shortcutting planned paths on the device (mpb200_shortcut_paths, planners.shortcut_paths): every output equals the CPU
restatement tests/oracle_shortcut.py byte for byte (length, states, cost, pairs, segment tests) on 2-D compounds (the
inverted point test included), N-d boxes up to 10-D and a position view, for paths from fmtstar, gmtstar and
gmtstar_batch and hand-made ones; the guarantees of the specification; independence from the rest of the call and the
grid; a fixed number of launches; the argument checks of the C ABI; C2 at full size."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import fixtures as fx
from oracle_shortcut import shortcut_oracle
from test_gpu_gmt import BOXES6D, _free_samples

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EARG, ENOMEM = -1, -4
KS = (1, 2, 4, 8)
BOXES10D = [np.array([[0.45, 0.55], [0.0, 0.6]] + [[0.0, 1.0]] * 8)]
PLANNED = ["ISRR_2H", "TRI_BALLS", "ISRR_POLY_WITH_SPIKE", "EMPTY_2D", "BOXES2D", "BOXES3D", "BOXES6D"]
HANDMADE = ["BOXES10D", "VIEW42"]


def _world(mp, orc, name):
    """-> (SS, CC, oracle obstacles, oracle space, d)"""
    if name in fx.ALL_2D:
        spec = fx.ALL_2D[name]
        return (mp.UnitHypercube(2), mp.PointRobot2D(fx.product_shape(mp, spec)), orc.Obstacles2D(spec),
                orc.StateSpace([0, 0], [1, 1]), 2)
    if name == "VIEW42":
        SS = mp.BoundedStateSpace(np.zeros(4), np.ones(4), mp.Euclidean(), mp.VectorView(1, 2))
        return (SS, mp.PointRobot2D(fx.product_shape(mp, fx.ISRR_2H)), orc.Obstacles2D(fx.ISRR_2H),
                orc.StateSpace([0] * 4, [1] * 4, ("view", [1, 2])), 4)
    boxes = {"BOXES2D": fx.BOXES2D, "BOXES3D": fx.BOXES3D, "BOXES6D": BOXES6D, "BOXES10D": BOXES10D}[name]
    d = boxes[0].shape[0]
    return (mp.UnitHypercube(d), mp.PointRobotNDBoxes([mp.BoxBounds(b) for b in boxes]), orc.Boxes(boxes),
            orc.StateSpace([0] * d, [1] * d), d)


def _planned_paths(mp, orc, name):
    """-> (SS, CC, O, So, [(states, planned cost)]) from fmtstar, gmtstar and gmtstar_batch over one sample set"""
    SS, CC, O, So, d = _world(mp, orc, name)
    N = 2000 if d == 2 else 3000
    V = _free_samples(orc, O, So, [0] * d, [1] * d, N, 20240601 if d == 2 else 7 + d, [0.1] * d, [0.9] * d)
    make = lambda: mp.MPProblem(SS, V[0], mp.PointGoal(V[-1]), CC, V=mp.MetricNN(V, SS.dist, V[0]))
    kw = dict(rm=1.5 if d == 3 else 1.2) if d > 2 else {}
    out = []
    P = make()
    mp.fmtstar(P, **kw)
    out.append((V[np.asarray(P.solution.metadata["path"]) - 1], P.solution.cost))
    P.V.close()
    P = make()
    mp.gmtstar(P, lam=1.0, **kw)
    out.append((V[np.asarray(P.solution.metadata["path"]) - 1], P.solution.cost))
    P.V.close()
    P = make()
    rng = np.random.Generator(np.random.PCG64(17))
    inits = [1] + [int(i) + 1 for i in rng.choice(N, 3, replace=False)]
    goals = [P.goal] + [mp.StateGoal(V[int(j)]) for j in rng.choice(N, 3, replace=False)]
    for s in mp.gmtstar_batch(P, inits, goals, lam=0.5, **kw):
        if s.status == "solved":
            out.append((V[np.asarray(s.metadata["path"]) - 1], s.cost))
    P.V.close()
    assert len(out) >= 3 and all(np.isfinite(c) for _, c in out)
    return SS, CC, O, So, out


def _handmade_paths(d, seed):
    """polylines in a region free by construction (x2 >= .65 beside the 10-D wall, x1 <= .2 before the 3-D boxes,
    y <= .18 below the 2-D sets), random ones (mostly blocked), one leaving the bounds and one single state"""
    rng = np.random.Generator(np.random.PCG64(seed))
    out = []
    for L in (2, 5, 9):
        Y = rng.random((L, d))
        if d == 10:
            Y[:, 1] = 0.65 + 0.35 * Y[:, 1]
        elif d == 3:
            Y[:, 0] = 0.2 * Y[:, 0]
        else:
            Y[:, 1] = 0.18 * Y[:, 1]
        out.append(Y)
    out += [rng.random((6, d)), rng.random((3, d))]
    Y = rng.random((4, d))
    Y[1, 0] = 1.25                                            # a waypoint outside the bounds: no segment test from it
    out.append(Y)
    out.append(rng.random((1, d)))
    return out


def _call(lib, CC, SS, paths, k, out_cap=None):
    """mpb200_shortcut_paths over `paths` -> (rc, [(out_len, states bytes or None, cost bytes, pairs, checks)])"""
    from mpb200 import _lib
    states = [np.ascontiguousarray(p, dtype=np.float64) for p in paths]
    n, d = len(states), states[0].shape[1]
    offs = np.zeros(n + 1, dtype=np.int64)
    offs[1:] = np.cumsum([len(s) for s in states])
    Y = np.ascontiguousarray(np.vstack(states))
    cap = max((len(s) - 1) * k + 1 for s in states) if out_cap is None else out_cap
    buf = np.full(n * cap * d + 64, -7.0)                     # exactly n x out_cap x d rows, then a guard
    out = buf[:n * cap * d].reshape(n, cap, d)
    out_len, costs = np.full(n, -1, dtype=np.int64), np.full(n, -1.0)
    pairs, segs = np.full(n, -1, dtype=np.int64), np.full(n, -1, dtype=np.int64)
    space = SS.desc()
    rc = lib.mpb200_shortcut_paths(_lib.ptr(Y), _lib.ptr(offs), n, d, CC.handle(), ctypes.byref(space), k,
                                   _lib.ptr(buf), cap, _lib.ptr(out_len), _lib.ptr(costs), _lib.ptr(pairs),
                                   _lib.ptr(segs))
    # nothing is written past a row's out_len, nothing into a row that does not fit, nothing past the rows
    assert np.all(buf[n * cap * d:] == -7.0)
    for q in range(n):
        assert np.all(out[q, max(int(out_len[q]), 0) if out_len[q] <= cap else 0:] == -7.0), q
    res = [(int(out_len[q]), out[q, :out_len[q]].tobytes() if 0 <= out_len[q] <= cap else None,
            costs[q].tobytes(), int(pairs[q]), int(segs[q])) for q in range(n)]
    return rc, res


def _expected(orc, O, So, Y, k):
    r = shortcut_oracle(orc, O, So, Y, k)
    return (len(r["states"]), np.ascontiguousarray(r["states"]).tobytes(), np.float64(r["cost"]).tobytes(),
            r["pairs"], r["segment_checks"])


def _states(res, d):
    return np.frombuffer(res[1], dtype=np.float64).reshape(-1, d)


@pytest.mark.parametrize("name", PLANNED)
def test_planned_paths_equal_the_restatement(gpu, orc, name):
    mp = gpu
    from mpb200 import _lib
    lib = _lib.lib()
    SS, CC, O, So, planned = _planned_paths(mp, orc, name)
    d = SS.dim
    paths = [Y for Y, _ in planned]
    for k in KS:
        rc, res = _call(lib, CC, SS, paths, k)
        assert rc == 0, lib.mpb200_last_error()
        for q, ((Y, planned_cost), r) in enumerate(zip(planned, res)):
            assert r == _expected(orc, O, So, Y, k), (k, q)
            S = _states(r, d)
            cost = np.frombuffer(r[2], dtype=np.float64)[0]
            assert cost <= planned_cost, (k, q)                                    # never above the planner's C[goal]
            assert np.array_equal(S[0], Y[0]) and np.array_equal(S[-1], Y[-1])
            assert len(S) < 2 or mp.segments_free(S[:-1], S[1:], CC, SS).all()     # free under an independent kernel
            rc2, again = _call(lib, CC, SS, [S], k)
            assert rc2 == 0 and np.frombuffer(again[0][2], dtype=np.float64)[0] <= cost


@pytest.mark.parametrize("name", HANDMADE + ["BOXES3D", "ISRR_POLY_WITH_SPIKE"])
def test_handmade_paths_equal_the_restatement(gpu, orc, name):
    mp = gpu
    from mpb200 import _lib
    lib = _lib.lib()
    SS, CC, O, So, d = _world(mp, orc, name)
    paths = _handmade_paths(d, 5 + d)
    for k in KS:
        rc, res = _call(lib, CC, SS, paths, k)
        assert rc == 0, lib.mpb200_last_error()
        for q, (Y, r) in enumerate(zip(paths, res)):
            assert r == _expected(orc, O, So, Y, k), (k, q)
            if np.isfinite(np.frombuffer(r[2], dtype=np.float64)[0]):
                S = _states(r, d)
                assert len(S) < 2 or mp.segments_free(S[:-1], S[1:], CC, SS).all()
            else:
                assert np.array_equal(_states(r, d), Y)                          # not free: the input unchanged
    assert any(np.isfinite(np.frombuffer(r[2], dtype=np.float64)[0]) and r[0] < len(Y) for Y, r in zip(paths, res))


def _batching_outputs(mp, orc, name, k):
    from mpb200 import _lib
    SS, CC, O, So, d = _world(mp, orc, name)
    paths = _handmade_paths(d, 3)
    rc, res = _call(_lib.lib(), CC, SS, paths, k)
    assert rc == 0
    return res


@pytest.mark.parametrize("name", ["ISRR_2H", "BOXES3D"])
def test_outputs_do_not_depend_on_the_rest_of_the_call(gpu, orc, name, tmp_path):
    mp = gpu
    from mpb200 import _lib
    lib = _lib.lib()
    SS, CC, O, So, d = _world(mp, orc, name)
    paths = _handmade_paths(d, 3)
    k = 4
    rc, base = _call(lib, CC, SS, paths, k)
    assert rc == 0
    for q, Y in enumerate(paths):
        rc, alone = _call(lib, CC, SS, [Y], k)
        assert rc == 0 and alone[0] == base[q], q
    rc, rev = _call(lib, CC, SS, paths[::-1], k)
    assert rc == 0 and rev[::-1] == base
    rc, mixed = _call(lib, CC, SS, paths[:2] + _handmade_paths(d, 99) + paths[2:], k)
    assert rc == 0 and mixed[:2] + mixed[2 + len(paths):] == base
    dump = str(tmp_path / "shortcut_child.npy")
    code = ("import sys, pickle; sys.path[:0] = [%r, %r]; import mpb200 as mp; mp.init(0)\n"
            "from oracle import oracle as orc; orc.lib()\n"
            "import test_gpu_shortcut as t\n"
            "pickle.dump(t._batching_outputs(mp, orc, %r, %d), open(%r, 'wb'))\n"
            % (ROOT, os.path.join(ROOT, "tests"), name, k, dump))
    subprocess.run([sys.executable, "-c", code], check=True, env=dict(os.environ, MPB200_SHORTCUT_GRID="3"), cwd=ROOT)
    import pickle
    with open(dump, "rb") as f:
        assert pickle.load(f) == base                                                # a three-CTA grid
    assert _batching_outputs(mp, orc, name, k) == base                              # and again, in this process


def test_launches_do_not_grow_with_the_number_of_paths(gpu, orc):
    mp = gpu
    from mpb200 import _lib
    lib = _lib.lib()
    SS, CC, O, So, d = _world(mp, orc, "ISRR_2H")
    paths = (_handmade_paths(d, 1) * 10)[:64]
    deltas = []
    for ps in (paths[:1], paths):
        before = lib.mpb200_launch_count()
        rc, _ = _call(lib, CC, SS, ps, 4)
        assert rc == 0
        deltas.append(lib.mpb200_launch_count() - before)
    assert deltas[0] == deltas[1] == 3


def test_argument_checks(gpu, orc):
    mp = gpu
    from mpb200 import _lib
    lib = _lib.lib()
    SS, CC, O, So, d = _world(mp, orc, "ISRR_2H")
    paths = _handmade_paths(d, 2)
    Y = np.ascontiguousarray(np.vstack(paths))
    offs = np.zeros(len(paths) + 1, dtype=np.int64)
    offs[1:] = np.cumsum([len(p) for p in paths])
    n, cap = len(paths), 64
    out = np.zeros((n, cap, d))
    ol, co, pa, sc = np.zeros(n, np.int64), np.zeros(n), np.zeros(n, np.int64), np.zeros(n, np.int64)
    space = SS.desc()
    P = _lib.ptr
    launches = lib.mpb200_launch_count()

    def rc(Yp=P(Y), o=P(offs), npaths=n, dd=d, cc=CC.handle(), sp=ctypes.byref(space), k=4, outp=P(out), oc=cap,
           olp=P(ol), cop=P(co)):
        return lib.mpb200_shortcut_paths(Yp, o, npaths, dd, cc, sp, k, outp, oc, olp, cop, P(pa), P(sc))

    assert rc(npaths=0) == EARG and rc(npaths=-2) == EARG
    for kw in (dict(Yp=None), dict(o=None), dict(olp=None), dict(cop=None)):
        assert rc(**kw) == EARG, kw
    for bad in (np.r_[1, offs[1:]], np.r_[offs[:2], offs[1], offs[2:-1]], np.r_[offs[:3], offs[2] - 1, offs[4:]]):
        assert rc(o=P(np.ascontiguousarray(bad, dtype=np.int64))) == EARG, bad   # not from 0 / an empty path / decreasing
    assert rc(k=0) == EARG and rc(k=-1) == EARG
    long_path = np.ascontiguousarray(np.linspace([0.05, 0.05], [0.06, 0.06], 4097))  # M = 4096 * 8 + 1 > 32768
    lo = np.array([0, 4097], dtype=np.int64)
    assert rc(Yp=P(long_path), o=P(lo), npaths=1, k=8) == EARG
    assert rc(outp=None) == EARG and rc(oc=-1) == EARG
    assert rc(cc=mp.PointRobotNDBoxes([mp.BoxBounds(b) for b in fx.BOXES3D]).handle()) == EARG  # 3-D boxes, 2-D space
    SS5 = mp.UnitHypercube(5)
    sp5 = SS5.desc()
    assert rc(dd=5, sp=ctypes.byref(sp5), o=P(np.array([0, 2], np.int64)), npaths=1) == EARG  # 2-D obstacles, d = 5
    assert rc(dd=3) == EARG                                                                  # space of another dimension
    assert lib.mpb200_launch_count() == launches                                             # no rejection launched
    # the limit itself is accepted; out_len is written even where the row does not fit
    edge = np.ascontiguousarray(np.linspace([0.05, 0.05], [0.06, 0.06], 32768))             # M = 32768 at k = 1
    rc1, r = _call(lib, CC, SS, [edge], 1, out_cap=1)
    assert rc1 == 0 and r[0][0] >= 2 and r[0][1] is None and r[0][3] == 32768 * 32767 // 2
    rc1, rows = _call(lib, CC, SS, paths, 4)
    short = _call(lib, CC, SS, paths, 4, out_cap=2)[1]
    assert [x[0] for x in short] == [x[0] for x in rows]
    assert all((s[1] is None) == (x[0] > 2) for s, x in zip(short, rows)) and any(x[0] > 2 for x in rows)
    assert all(s[1] == x[1] for s, x in zip(short, rows) if x[0] <= 2)
    assert lib.mpb200_shortcut_paths(P(Y), P(offs), n, d, CC.handle(), ctypes.byref(space), 4, None, 0, P(ol), P(co),
                                     None, None) == 0                                 # out_cap = 0 with no rows
    assert [int(x) for x in ol] == [x[0] for x in rows]


def test_python_api(gpu, orc):
    mp = gpu
    SS, CC, O, So, d = _world(mp, orc, "ISRR_2H")
    V = _free_samples(orc, O, So, [0, 0], [1, 1], 2000, 20240603, [0.1, 0.1], [0.9, 0.9])
    P = mp.MPProblem(SS, V[0], mp.PointGoal(V[-1]), CC, V=mp.MetricNN(V, SS.dist, V[0]))
    mp.gmtstar(P, lam=1.0)
    before = CC.count
    (r,) = mp.shortcut_paths(P)
    ref = shortcut_oracle(orc, O, So, V[np.asarray(P.solution.metadata["path"]) - 1], 4)
    assert r["states"].tobytes() == ref["states"].tobytes() and r["cost"] == ref["cost"] <= P.solution.cost
    assert (r["pairs"], r["segment_checks"]) == (ref["pairs"], ref["segment_checks"])
    assert CC.count - before == r["segment_checks"]
    r2, r3 = mp.shortcut_paths(P, [P.solution.metadata["path"], r["states"]], subdivisions=2)
    assert r3["cost"] <= r["cost"] and np.array_equal(r2["states"][[0, -1]], r["states"][[0, -1]])
    for bad in ([[]], [[0, 1]], [[1, len(V) + 1]], [np.zeros((3, 3))]):
        with pytest.raises(ValueError):
            mp.shortcut_paths(P, bad)
    with pytest.raises(ValueError):
        mp.shortcut_paths(P, subdivisions=0)
    P.V.close()
    for SSc in (mp.ReedsSheppMetricSpace(0.05, 1.0), mp.DubinsQuasiMetricSpace(0.05, 1.0), mp.DoubleIntegrator(2)):
        Pc = mp.MPProblem(SSc, SSc.lo + 0.1, mp.StateGoal(SSc.lo + 0.2), CC)
        with pytest.raises(ValueError):
            mp.shortcut_paths(Pc, [np.vstack([SSc.lo + 0.1, SSc.lo + 0.2])])


def test_full_size_c2_equals_the_restatement(gpu, orc):
    """C2 (ISRR_2H, N = 1M, seed 20240602, lambda = 1): 4 gmtstar_batch queries shortcut at k = 4"""
    mp = gpu
    from mpb200 import _lib
    N = 1_000_000
    SS = mp.UnitHypercube(2)
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    P = mp.MPProblem(SS, [0.1, 0.1], mp.BallGoal([0.9, 0.9], 0.01), CC)
    rng = np.random.Generator(np.random.PCG64(2024))
    inits = [1] + [int(i) for i in rng.integers(2, N + 1, 7)]          # sample_free draws free states only
    goals = [P.goal] + [mp.BallGoal(c, 0.01) for c in rng.random((7, 2))]
    sols = mp.gmtstar_batch(P, inits, goals, lam=1.0, N=N, seed=20240602, trees=False)
    V = P.V.V
    solved = [s for s in sols if s.status == "solved"]
    assert len(solved) >= 4
    paths = [V[np.asarray(s.metadata["path"]) - 1] for s in solved[:4]]
    rc, res = _call(_lib.lib(), CC, SS, paths, 4)
    assert rc == 0
    O, So = orc.Obstacles2D(fx.ISRR_2H), orc.StateSpace([0, 0], [1, 1])
    for Y, s, r in zip(paths, solved, res):
        assert r == _expected(orc, O, So, Y, 4)
        assert np.frombuffer(r[2], dtype=np.float64)[0] <= s.cost
    P.V.close()
