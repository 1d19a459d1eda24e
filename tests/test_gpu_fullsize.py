"""GPU parity at BASELINE.json's FULL sizes for the secondary configs (C3: 10-D, N = 2M; C4: double
integrator, N = 200k) and the adversarial cases of the tensor-core prefilter's error band in 10-D.
The oracle is run on column windows spread over the index range (it cannot do 4e12 pairs); the device
tables are compared byte for byte on those windows through device views (the 15 GB table is never copied)."""
import numpy as np
import pytest

import fixtures as fx
from conftest import unpack_bits

pytestmark = pytest.mark.gpu


def _device_columns(table, a, b):
    """(colptr - colptr[a], rowval, nzval, first entry) of columns [a, b) of a device table"""
    from mpb200 import sharding
    colptr, rowval, nzval, _ = sharding.table_device_tensors(table)
    cp = colptr[a:b + 1].cpu().numpy()
    lo, hi = int(cp[0]) - 1, int(cp[-1]) - 1
    return cp - cp[0], rowval[lo:hi].cpu().numpy(), nzval[lo:hi].cpu().numpy(), lo


def _same_columns(dev, ref):
    return (np.array_equal(dev[0], ref[0] - ref[0][0]) and np.array_equal(dev[1], ref[1])
            and dev[2].tobytes() == np.ascontiguousarray(ref[2]).tobytes())


def test_full_size_c3_table_and_box_edges(gpu, orc):
    """BASELINE config 3: 10-D unit hypercube, 64 random hyperboxes (seed 20240613), N = 2M, FMT* radius:
    tcgen05 prefilter + exact recheck, then box edge validity -- 8 windows x 16 query columns over the index range."""
    mp = gpu
    d, N = 10, 2_000_000
    V = fx.uniform_samples(N, d, 20240603)
    r = fx.fmt_radius(N, d)
    boxes = fx.random_hyperboxes(64, d, 20240613)
    CC = mp.PointRobotNDBoxes([mp.BoxBounds(*b) for b in boxes])
    SS = mp.UnitHypercube(d)
    B = orc.Boxes(boxes)
    So = orc.StateSpace(np.zeros(d), np.ones(d))
    NN = mp.MetricNN(V)
    nnz = NN.build_table(r)
    assert 400 * N < nnz < 600 * N                       # mean degree ~487 (SURVEY 8d)
    bits, checks = NN.edges_free(NN.table, CC, SS)
    assert checks == nnz
    got = unpack_bits(bits, nnz)
    cols = 0
    for a in np.linspace(0, N - 16, 8).astype(np.int64):
        a = int(a)
        ref = orc.rball_brute(V, r, 0, a, a + 16)
        dev = _device_columns(NN.table, a, a + 16)
        assert _same_columns(dev, ref), "columns [%d, %d)" % (a, a + 16)
        exp, _ = orc.edges_free_csc(B, So, V, ref[0], ref[1], a)
        assert np.array_equal(got[dev[3]:dev[3] + len(ref[1])], exp.astype(bool))
        cols += 16
    assert cols == 128
    assert 0 < int((~got).sum()) < nnz                     # both outcomes occur (hyperboxes are thin in 10-D: ~0.1% collide)
    NN.close()


def test_full_size_c4_lq_tables_and_edges(gpu, orc):
    """BASELINE config 4: double integrator (4-D state), N = 200k, ControlNN tables in both directions and the
    swept LQ edge validity of the backward table -- 4 windows x 16 columns per direction."""
    mp = gpu
    N = 200_000
    rng = np.random.Generator(np.random.PCG64(20240604))
    SS = mp.DoubleIntegrator(2)
    V = SS.lo + rng.random((N, 4)) * (SS.hi - SS.lo)
    r = 0.69                                              # mean degree ~64 at N = 200k (SURVEY 8d)
    L = orc.DoubleIntegratorLQ(2)
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    O = orc.Obstacles2D(fx.ISRR_2H)
    C = np.hstack([np.eye(2), np.zeros((2, 2))])
    So = orc.StateSpace(SS.lo, SS.hi, ("matrix", C))
    NN = mp.QuasiMetricNN(V, SS.dist)
    nF, nB = NN.build_tables(r)
    assert nF == nB and 30 * N < nB < 120 * N
    bits, checks = NN.lq_edges_free(CC, SS)
    got = unpack_bits(bits, nB)
    cols = 0
    for a in np.linspace(0, N - 16, 4).astype(np.int64):
        a = int(a)
        for forwards, table in ((True, NN.tableF), (False, NN.tableB)):
            ref = L.inball(V, r, forwards, a, a + 16)
            dev = _device_columns(table, a, a + 16)
            assert _same_columns(dev, ref), "%s columns [%d, %d)" % ("F" if forwards else "B", a, a + 16)
            cols += 16
            if not forwards:
                exp, _ = L.edges_free_csc(O, So, r, V, ref[0], ref[1], a)
                assert np.array_equal(got[dev[3]:dev[3] + len(ref[1])], np.asarray(exp).astype(bool))
    assert cols == 128
    NN.close()


@pytest.mark.parametrize("offset", [0.0, 1000.0, -3.0e4])
def test_k3_tensor_core_band_adversarial_10d(gpu, orc, offset):
    """d = 10, compact cloud (the tensor-core prefilter is in use): partners planted EXACTLY at the radius along
    several lattice directions, partners one ulp-scale step beyond it, and the whole cloud translated far from
    the origin (the TF32 operands are formed after centring).  Sets and distances byte-equal to the brute oracle."""
    mp = gpu
    rng = np.random.Generator(np.random.PCG64(2718))
    d, step = 10, 1.0 / 32
    base = fx.lattice_cloud(rng, 700, d, step, 0.0, 0.65)
    r = 10.0 / 32                                          # |(6,8,0..)|/32 = |(5,5,5,5,0..)|/32 = |(4,4,4,4,4,4,2,0..)|/32
    dirs = np.zeros((3, d))
    dirs[0, :2] = (6, 8)
    dirs[1, 2:6] = 5
    dirs[2, :6] = 4
    dirs[2, 6] = 2
    at_r = [base + dirs[k] * step for k in range(3)]
    beyond = base + dirs[0] * step
    beyond[:, 9] += 2.0 ** -20                             # s = r^2 + 2^-40: not a member, deep inside the TF32 band
    inside = base + dirs[1] * step
    inside[:, 2] -= 2.0 ** -20                             # s just below r^2
    W = np.vstack([base] + at_r + [beyond, inside]) + offset
    NN = mp.MetricNN(W)
    D = NN.precompute(r).D
    ref = orc.rball_brute(W, r)
    assert np.array_equal(D.colptr, ref[0]) and np.array_equal(D.rowval, ref[1])
    assert D.nzval.tobytes() == ref[2].tobytes()
    if offset == 0.0:
        assert (D.nzval == r).sum() >= 2 * 3 * 700         # every planted exactly-at-radius pair is stored (both directions)
    NN.close()


def test_k3_wide_sparse_cloud_small_radius_takes_the_cuda_core_path(gpu, orc):
    """A wide cloud with a tiny radius: the TF32 allowance is not small against r^2, so the build must not rely
    on the tensor-core band (brute_rball.cu: tc_band_is_tight) -- and the result is exact either way."""
    mp = gpu
    rng = np.random.Generator(np.random.PCG64(99))
    d = 10
    base = rng.random((1500, d)) * 2000.0 - 1000.0
    r = 1e-3
    near = base[:600] + rng.standard_normal((600, d)) * (r / 4.0)    # partners well inside / around the radius
    exact = base[600:1200].copy()
    exact[:, 0] = np.round(exact[:, 0] * 1024) / 1024
    partner = exact.copy()
    partner[:, 0] += 2.0 ** -10                                      # distance exactly 2^-10 < r ... a member
    W = np.vstack([base[:600], near, exact, partner, base[1200:]])
    NN = mp.MetricNN(W)
    D = NN.precompute(r).D
    ref = orc.rball_brute(W, r)
    assert np.array_equal(D.colptr, ref[0]) and np.array_equal(D.rowval, ref[1])
    assert D.nzval.tobytes() == ref[2].tobytes()
    assert D.nnz >= 2 * 600
    NN.close()


@pytest.mark.parametrize("kind", ["reedsshepp", "dubins"])
def test_f4_car_tables_at_bench_size(gpu, orc, kind):
    """bench config F4 (N = 200k SE2 states, turning radius 0.01, r = 0.025): 96 columns in three windows of the index
    range, both directions for Dubins, and the arc-waypoint edge bits of those columns, byte for byte"""
    import math
    mp = gpu
    N, rturn, r = 200_000, 0.01, 0.025
    rng = np.random.Generator(np.random.PCG64(20240605))
    V = np.column_stack([rng.random(N), rng.random(N), rng.uniform(0, 2 * math.pi, N)])
    SS = (mp.ReedsSheppMetricSpace if kind == "reedsshepp" else mp.DubinsQuasiMetricSpace)(rturn)
    mp.setup_steering(SS, r)
    car = orc.SimpleCar(kind, rturn)
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    O = orc.Obstacles2D(fx.ISRR_2H)
    So = orc.StateSpace(SS.lo, SS.hi, ("view", [1, 2]))
    if kind == "reedsshepp":
        NN = mp.MetricNN(V, SS.dist, V[0])
        tables = [(NN.precompute(r).D, True)]
    else:
        NN = mp.QuasiMetricNN(V, SS.dist, V[0])
        cF, cB = NN.precompute(r)
        tables = [(cF.D, True), (cB.D, False)]
    bits, _ = NN.car_edges_free(CC, SS)
    Dlast = tables[-1][0]                                # the table the edge bits belong to
    ebits = unpack_bits(bits, Dlast.nnz)
    for q0 in (0, N // 2 - 16, N - 32):
        for D, fw in tables:
            ref = car.inball(V, r, fw, q0=q0, q1=q0 + 32)
            lo, hi = D.colptr[q0] - 1, D.colptr[q0 + 32] - 1
            assert np.array_equal(D.colptr[q0:q0 + 33] - D.colptr[q0], ref[0] - 1)
            assert np.array_equal(D.rowval[lo:hi], ref[1]) and D.nzval[lo:hi].tobytes() == ref[2].tobytes()
        exp, _ = car.edges_free_csc(O, So, V, ref[0], ref[1], c0=q0)
        assert np.array_equal(ebits[lo:hi], exp.astype(bool))
    NN.close()
