"""Roadmap-optimal plans on the device (mpb200_sssp_plan through planners.prmstar): every output equals the CPU
restatement tests/oracle_sssp.py over the same fetched tables and bits on the eight problem kinds of test_gpu_gmt.py,
with and without checkpts, and on sets with duplicated samples and tied lattice costs; DF holds the transpose of DB;
PRM* is never worse than GMT* over the same roadmap; outputs do not depend on the grid; one launch per plan;
shortcutting a PRM* path; C2 at full size; the argument checks of the C ABI."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import fixtures as fx
from oracle_sssp import sssp_numpy, sssp_oracle
from test_gpu_gmt import CASES, _case, _tables_of, fx_bits

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EARG = -1


def _oracle_over(P, B_tab, ebits, checkpts=True, numpy=False):
    from mpb200.problems import goal_mask
    N = len(P.V)
    free = fx_bits(P.V.points_free(P.CC, P.SS), N) if checkpts else np.ones(N, dtype=bool)
    f = sssp_numpy if numpy else sssp_oracle
    return f(N, B_tab.colptr, B_tab.rowval, B_tab.nzval, ebits, free, goal_mask(P.V.V, P.goal, P.SS))


def _assert_equal(m, st, cost, ref):
    assert (st == "solved") == ref["solved"]
    assert np.float64(cost).tobytes() == np.float64(ref["cost"]).tobytes()
    assert m["path"] == ref["path"] and np.array_equal(m["tree"], ref["tree"])
    assert m["costs"].tobytes() == ref["costs"].tobytes()
    assert (m["reached"], m["levels"]) == (ref["reached"], ref["levels"])
    assert m["planner"] == "PRMstar"


def _transpose_included(F_tab, B_tab):
    """every entry (row y, column x) of DB has x in column y of DF"""
    N = len(B_tab.colptr) - 1
    bcol = np.repeat(np.arange(N), np.diff(B_tab.colptr))
    fcol = np.repeat(np.arange(N), np.diff(F_tab.colptr))
    need = set(zip((np.asarray(B_tab.rowval) - 1).tolist(), bcol.tolist()))          # (y, x): x in DF column y
    have = set(zip(fcol.tolist(), (np.asarray(F_tab.rowval) - 1).tolist()))
    return need <= have


@pytest.mark.parametrize("name", CASES)
def test_prm_equals_the_cpu_restatement_and_dominates_gmt(gpu, orc, name):
    mp = gpu
    make, kw = _case(mp, orc, name)
    P = make()
    for checkpts in (True, False):
        st, cost, _ = mp.prmstar(P, checkpts=checkpts, **kw)
        m = P.solution.metadata
        F_tab, B_tab, ebits = _tables_of(P.V, name, kw)
        assert _transpose_included(F_tab, B_tab)
        ref = _oracle_over(P, B_tab, ebits, checkpts)
        assert ref["solved"]
        _assert_equal(m, st, cost, ref)
        # the parent chain folds to the cost, bit for bit
        c = 0.0
        for y, x in zip(m["path"][:-1], m["path"][1:]):
            lo, hi = B_tab.colptr[x - 1] - 1, B_tab.colptr[x] - 1
            c = c + float(B_tab.nzval[lo + int(np.flatnonzero(B_tab.rowval[lo:hi] == y)[0])])
        assert c == cost
    # GMT* over the same roadmap never beats it
    st_p, cost_p, _ = mp.prmstar(P, **kw)
    d = P.solution.metadata["costs"].copy()
    for lam in (0.0, 0.5, 1.0, 4.0):
        st_g, cost_g, _ = mp.gmtstar(P, lam=lam, **kw)
        mg = P.solution.metadata
        if st_g == "solved":
            assert st_p == "solved" and cost_p <= cost_g, lam
        reached = (mg["tree"] != 0)
        reached[0] = True
        in_r = np.isfinite(d)
        assert np.all(d[reached & in_r] <= mg["costs"][reached & in_r]), lam
    P.V.close()


def _tie_sets(mp, kind):
    """2-D sets where zero-cost entries and ties reach the kernel: samples duplicated (the same state twice), and a
    lattice whose equal spacing ties many routes"""
    SS = mp.UnitHypercube(2)
    CC = mp.PointRobot2D(fx.product_shape(mp, fx.ISRR_2H))
    rng = np.random.Generator(np.random.PCG64(5))
    if kind == "duplicates":
        V = rng.random((1500, 2))
        V = np.vstack([[0.1, 0.1], V, V[rng.choice(1500, 500, replace=False)], [0.9, 0.9]])
        r = 0.06
    else:
        g = np.linspace(0.0, 1.0, 41)
        V = np.stack(np.meshgrid(g, g, indexing="ij"), -1).reshape(-1, 2)
        V = np.vstack([[0.1, 0.1], V, [0.9, 0.9]])
        r = 0.051
    return lambda: mp.MPProblem(SS, V[0], mp.PointGoal(V[-1]), CC, V=mp.MetricNN(V, SS.dist, V[0])), dict(r=r)


@pytest.mark.parametrize("kind", ["duplicates", "lattice"])
def test_prm_with_zero_cost_entries_and_ties(gpu, kind):
    mp = gpu
    make, kw = _tie_sets(mp, kind)
    P = make()
    for checkpts in (True, False):
        st, cost, _ = mp.prmstar(P, checkpts=checkpts, **kw)
        F_tab, B_tab, ebits = _tables_of(P.V, kind, kw)
        if kind == "duplicates":
            assert np.any(B_tab.nzval == 0.0)
        ref = _oracle_over(P, B_tab, ebits, checkpts)
        _assert_equal(P.solution.metadata, st, cost, ref)
    P.V.close()


def _plan_outputs(mp, make, kw):
    P = make()
    mp.prmstar(P, **kw)
    m = P.solution.metadata
    out = (m["tree"].tobytes(), m["costs"].tobytes(), tuple(m["path"]), np.float64(m["cost"]).tobytes(),
           m["rounds"], m["levels"], m["reached"])
    P.V.close()
    return out, m["grid_blocks"]


def test_prm_is_deterministic_across_runs_and_grid_sizes(gpu, orc, tmp_path):
    mp = gpu
    make, kw = _case(mp, orc, "2d_20k")
    a, blocks = _plan_outputs(mp, make, kw)
    b, _ = _plan_outputs(mp, make, kw)
    assert a == b
    dump = str(tmp_path / "sssp_child.npz")
    code = ("import sys, numpy as np; sys.path[:0] = [%r, %r]; import mpb200 as mp; mp.init(0)\n"
            "from oracle import oracle as orc; orc.lib()\n"
            "import test_gpu_gmt as g, test_gpu_sssp as t\n"
            "make, kw = g._case(mp, orc, '2d_20k')\n"
            "o, blocks = t._plan_outputs(mp, make, kw)\n"
            "np.savez(%r, blocks=blocks, **{'o%%d' %% i: np.frombuffer(x, np.uint8) if isinstance(x, bytes) else np.asarray(x) for i, x in enumerate(o)})\n"
            % (ROOT, os.path.join(ROOT, "tests"), dump))
    env = dict(os.environ, MPB200_GMT_GRID="37")
    subprocess.run([sys.executable, "-c", code], check=True, env=env, cwd=ROOT)
    with np.load(dump) as z:
        assert int(z["blocks"]) == 37 != blocks
        for i, x in enumerate(a):
            got = z["o%d" % i]
            assert (got.tobytes() == x) if isinstance(x, bytes) else np.array_equal(got, np.asarray(x)), i


def _sssp_call(NN, DF, DB, goal_mask_bool, init=1, checkpts=1, path_cap=None):
    from mpb200 import _lib
    N = len(NN)
    chunks = np.zeros((N + 63) // 64 * 8, dtype=np.uint8)
    pk = np.packbits(goal_mask_bool, bitorder="little")
    chunks[:len(pk)] = pk
    chunks = chunks.view(np.uint64)
    desc = _lib.GmtDesc(DF.h if DF is not None else None, DB.h if DB is not None else None, _lib.ptr(chunks), init,
                        0.0, checkpts, None)
    res = _lib.SsspResult()
    cap = N if path_cap is None else path_cap
    path = np.full(max(cap, 1), -7, dtype=np.int64)
    rc = _lib.lib().mpb200_sssp_plan(NN.handle(), ctypes.byref(desc), ctypes.byref(res), _lib.ptr(path), cap, None,
                                     None)
    return rc, res, path


def test_prm_launches_once_per_plan_and_checks_its_arguments(gpu, orc):
    mp = gpu
    lib = mp.load()
    make, kw = _case(mp, orc, "2d_2k")
    P = make()
    mp.prmstar(P, **kw)
    NN = P.V
    from mpb200.problems import goal_mask
    goal = goal_mask(NN.V, P.goal, P.SS)
    for g in (goal, np.zeros(len(NN), dtype=bool)):                # solved, and the full tree
        before = lib.mpb200_launch_count()
        rc, res, path = _sssp_call(NN, NN.table, NN.table, g)
        assert rc == 0 and lib.mpb200_launch_count() - before == 1
    assert not res.solved and res.reached > 0
    rc, res, path = _sssp_call(NN, NN.table, NN.table, goal)
    assert rc == 0 and res.solved and list(path[:res.path_len]) == P.solution.metadata["path"]
    rc, res2, path = _sssp_call(NN, NN.table, NN.table, goal, path_cap=res.path_len - 1)  # path_cap too small
    assert rc == 0 and res2.path_len == res.path_len and np.all(path == -7)
    SS, CC = P.SS, P.CC
    other = mp.MetricNN(NN.V.copy())                                   # same N and d, another sample set
    other.build_table_checked(0.05, CC, SS)
    assert _sssp_call(NN, other.table, NN.table, goal)[0] == EARG
    assert _sssp_call(NN, NN.table, other.table, goal)[0] == EARG
    other.close()
    assert _sssp_call(NN, NN.table, NN.table, goal, init=0)[0] == EARG
    assert _sssp_call(NN, NN.table, NN.table, goal, init=len(NN) + 1)[0] == EARG
    assert _sssp_call(NN, None, NN.table, goal)[0] == EARG
    NN.build_table(0.05)                                                # new contents, stale edge bits
    assert _sssp_call(NN, NN.table, NN.table, goal)[0] == EARG
    NN.edges_free(NN.table, CC, SS, fetch=False)
    assert _sssp_call(NN, NN.table, NN.table, goal)[0] == 0
    fresh = mp.MetricNN(NN.V.copy())                                    # no point bits yet
    fresh.build_table_checked(0.05, CC, SS)
    assert _sssp_call(fresh, fresh.table, fresh.table, goal)[0] == EARG
    assert _sssp_call(fresh, fresh.table, fresh.table, goal, checkpts=0)[0] == 0
    fresh.set_query_range(0, 1000)                                      # point bits of a shard only
    fresh.points_free(CC, SS, fetch=False)
    assert _sssp_call(fresh, fresh.table, fresh.table, goal)[0] == EARG
    fresh.build_table_checked(0.05, CC, SS)                             # a sharded table
    assert _sssp_call(fresh, fresh.table, fresh.table, goal, checkpts=0)[0] == EARG
    fresh.close()
    NN.close()


def test_shortcut_of_a_prm_path_is_no_costlier(gpu, orc):
    mp = gpu
    make, kw = _case(mp, orc, "2d_2k")
    P = make()
    st, cost, _ = mp.prmstar(P, **kw)
    assert st == "solved"
    out = mp.shortcut_paths(P, subdivisions=4)
    assert out[0]["cost"] <= cost
    P.V.close()


def test_prm_full_size_c2_matches_the_numpy_restatement(gpu):
    """C2 (ISRR_2H, N = 1M, r from fmt_radius) against the frontier restatement over the fetched table"""
    mp = gpu
    N = 1_000_000
    SS = mp.UnitHypercube(2)
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    P = mp.MPProblem(SS, [0.1, 0.1], mp.BallGoal([0.9, 0.9], 0.01), CC)
    st, cost, _ = mp.prmstar(P, N, seed=20240602)
    m = P.solution.metadata
    NN = P.V
    T = NN.fetch_table(NN.table)
    from mpb200 import _lib
    bits = np.empty((T.nnz + 63) // 64, dtype=np.uint64)
    _lib.check(_lib.lib().mpb200_table_fetch_edge_bits(NN.table.h, _lib.ptr(bits)))
    ref = _oracle_over(P, T, fx_bits(bits, T.nnz), numpy=True)
    assert st == "solved" and ref["solved"]
    assert np.float64(cost).tobytes() == np.float64(ref["cost"]).tobytes() and m["path"] == ref["path"]
    assert m["costs"].tobytes() == ref["costs"].tobytes() and np.array_equal(m["tree"], ref["tree"])
    assert (m["reached"], m["levels"]) == (ref["reached"], ref["levels"])
    NN.close()
