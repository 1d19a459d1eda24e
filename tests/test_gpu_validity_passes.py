"""Point validity (K6) and edge validity (K7/K8) over r-ball tables, against the CPU oracle.

After a grid build the point pass reads the build's cell-ordered copy of the samples, and the edge pass on a
Euclidean r-ball table classifies whole columns and runs the per-edge test on the rest in one launch.  These cases
drive both through every layout they handle: full sets and shards, 2-D compounds of each kind and N-d boxes, tables
with and without a cell order, ragged column counts, long and empty columns, and copies that no longer describe
the table."""
import numpy as np
import pytest

import fixtures as fx
from conftest import unpack_bits

pytestmark = pytest.mark.gpu

BENCH_SEED = 20240602


def _checker(mp, orc, name):
    if name == "BOXES3D":
        return mp.PointRobotNDBoxes([mp.BoxBounds(b) for b in fx.BOXES3D]), orc.Boxes(fx.BOXES3D)
    if name == "RANDOM10":
        bl = fx.random_hyperboxes(64, 10, 20240613)
        return (mp.PointRobotNDBoxes([mp.BoxBounds(*b) if isinstance(b, tuple) else mp.BoxBounds(b) for b in bl]),
                orc.Boxes(bl))
    spec = fx.ALL_2D[name]
    return mp.PointRobot2D(fx.product_shape(mp, spec)), orc.Obstacles2D(spec)


def _spaces(mp, orc, d):
    lo, hi = np.zeros(d), np.ones(d)
    return mp.BoundedStateSpace(lo, hi, mp.Euclidean(), mp.Identity()), orc.StateSpace(lo, hi)


def _check_points(orc, NN, CC, R, SSp, SSo, V, q0=0, q1=None):
    q1 = len(V) if q1 is None else q1
    got = unpack_bits(NN.points_free(CC, SSp), q1 - q0)
    assert np.array_equal(got, orc.states_free(R, SSo, V[q0:q1]).astype(bool))


def _check_edges(orc, NN, table, CC, R, SSp, SSo, V, q0=0):
    D = NN.fetch_table(table)
    bits, checks = NN.edges_free(table, CC, SSp)
    exp, cnt = orc.edges_free_csc(R, SSo, V, D.colptr, D.rowval, q0)
    got = unpack_bits(bits, D.nnz)
    assert np.array_equal(got, exp.astype(bool))
    assert checks == cnt
    if D.nnz % 64:
        assert int(bits[-1]) >> (D.nnz % 64) == 0      # unused high bits of the last chunk stay zero
    return D, got, cnt


@pytest.mark.parametrize("N", [200_000, 1_000_000])
def test_isrr_2h_bench_samples(gpu, orc, N):
    """the flagship set (ISRR_2H, unit square, bench seed and radius) -- every point bit and every edge bit"""
    mp = gpu
    V = fx.uniform_samples(N, 2, BENCH_SEED)
    r = fx.fmt_radius(N, 2)
    CC, R = _checker(mp, orc, "ISRR_2H")
    SSp, SSo = _spaces(mp, orc, 2)
    NN = mp.MetricNN(V)
    NN.build_table(r)
    _check_points(orc, NN, CC, R, SSp, SSo, V)
    D, got, cnt = _check_edges(orc, NN, NN.table, CC, R, SSp, SSo, V)
    assert D.nnz > 20 * N
    # the build with the edge pass fused reports the same bits and count
    nnz, checks = NN.build_table_checked(r, CC, SSp)
    assert nnz == D.nnz and checks == cnt
    assert np.array_equal(unpack_bits(NN.fetch_edge_bits(), D.nnz), got)
    NN.close()


@pytest.mark.parametrize("name", ["TRI_BALLS", "ISRR_POLY", "EMPTY_2D", "ISRR_POLY_WITH_SPIKE"])
def test_2d_compounds(gpu, orc, name):
    """circles (no polygon fast path), polygons, the empty set; samples partly outside the bounds"""
    mp = gpu
    N = 60_013                                            # ncols not a multiple of 32
    V = fx.uniform_samples(N, 2, 11) * 1.04 - 0.02
    CC, R = _checker(mp, orc, name)
    SSp, SSo = _spaces(mp, orc, 2)
    NN = mp.MetricNN(V)
    NN.build_table(fx.fmt_radius(N, 2))
    _check_points(orc, NN, CC, R, SSp, SSo, V)
    _check_edges(orc, NN, NN.table, CC, R, SSp, SSo, V)
    NN.close()


@pytest.mark.parametrize("name,d,N", [("BOXES3D", 3, 40_007), ("RANDOM10", 10, 6_001)])
def test_nd_boxes(gpu, orc, name, d, N):
    """3-D boxes over a grid table (cell order) and 10-D boxes over an all-pairs table (no cell order)"""
    mp = gpu
    V = fx.uniform_samples(N, d, 23 + d) * 1.04 - 0.02
    r = fx.fmt_radius(N, d) * (1.0 if d == 3 else 1.3)
    CC, R = _checker(mp, orc, name)
    SSp, SSo = _spaces(mp, orc, d)
    NN = mp.MetricNN(V)
    NN.build_table(r)
    _check_points(orc, NN, CC, R, SSp, SSo, V)
    D, _, _ = _check_edges(orc, NN, NN.table, CC, R, SSp, SSo, V)
    assert D.nnz > N
    NN.close()


@pytest.mark.parametrize("name,d", [("ISRR_2H", 2), ("ISRR_POLY", 2), ("BOXES3D", 3)])
def test_shard(gpu, orc, name, d):
    """a query range with q0 > 0: columns start at col0 != 0 and the cell-order walk goes through q_order"""
    mp = gpu
    N = 50_000
    V = fx.uniform_samples(N, d, 41 + d)
    CC, R = _checker(mp, orc, name)
    SSp, SSo = _spaces(mp, orc, d)
    q0, q1 = 12_345, 37_001
    NN = mp.MetricNN(V)
    NN.set_query_range(q0, q1)
    NN.build_table(fx.fmt_radius(N, d))
    _check_points(orc, NN, CC, R, SSp, SSo, V, q0, q1)
    D, _, _ = _check_edges(orc, NN, NN.table, CC, R, SSp, SSo, V, q0)
    assert len(D.colptr) == q1 - q0 + 1
    NN.close()


@pytest.mark.parametrize("r", [0.06, 1e-4])
def test_long_and_empty_columns(gpu, orc, r):
    """large r: every column well over 32 entries (several rounds of the per-edge loop); tiny r: nearly all
    columns empty"""
    mp = gpu
    N = 20_011
    V = fx.uniform_samples(N, 2, 5)
    CC, R = _checker(mp, orc, "ISRR_POLY")
    SSp, SSo = _spaces(mp, orc, 2)
    NN = mp.MetricNN(V)
    NN.build_table(r)
    D, _, _ = _check_edges(orc, NN, NN.table, CC, R, SSp, SSo, V)
    deg = np.diff(D.colptr)
    if r > 0.01:
        assert deg.min() > 32
    else:
        assert (deg == 0).mean() > 0.9
    _check_points(orc, NN, CC, R, SSp, SSo, V)
    NN.close()


@pytest.mark.parametrize("name,d", [("ISRR_2H", 2), ("BOXES3D", 3)])
def test_points_and_edges_across_builds(gpu, orc, name, d):
    """points before any build, after a build, and after a build of another radius; edges of a table whose
    samples have since been rebuilt at another radius (its cell-ordered copy is gone) and after a query-range
    change"""
    mp = gpu
    N = 30_011
    V = fx.uniform_samples(N, d, 77 + d) * 1.06 - 0.03
    CC, R = _checker(mp, orc, name)
    SSp, SSo = _spaces(mp, orc, d)
    r = fx.fmt_radius(N, d)
    NN = mp.MetricNN(V)
    _check_points(orc, NN, CC, R, SSp, SSo, V)                  # no grid yet: index order
    NN.build_table(r)
    first = NN.table
    _check_points(orc, NN, CC, R, SSp, SSo, V)
    _check_edges(orc, NN, first, CC, R, SSp, SSo, V)
    NN.table = type(first)("other")
    NN.build_table(1.5 * r)                                 # the samples' grid now belongs to this table
    _check_points(orc, NN, CC, R, SSp, SSo, V)
    _check_edges(orc, NN, NN.table, CC, R, SSp, SSo, V)
    _check_edges(orc, NN, first, CC, R, SSp, SSo, V)        # stale copy: the pass must gather from V
    NN.set_query_range(0, N // 2)                           # the copy no longer matches the query range
    _check_points(orc, NN, CC, R, SSp, SSo, V, 0, N // 2)
    _check_edges(orc, NN, NN.table, CC, R, SSp, SSo, V)
    first.close()
    NN.close()
