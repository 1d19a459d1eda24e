"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same seeded
inputs -- bit-exact booleans and neighbour sets, exactly equal distances."""
import numpy as np
import pytest

import fixtures as fx
from conftest import unpack_bits

pytestmark = pytest.mark.gpu


def _space_pair(mp, orc, lo, hi, s2w=None):
    if s2w is None:
        return mp.BoundedStateSpace(lo, hi, mp.Euclidean(), mp.Identity()), orc.StateSpace(lo, hi)
    if s2w[0] == "view":
        return mp.BoundedStateSpace(lo, hi, mp.Euclidean(), mp.VectorView(s2w[1])), orc.StateSpace(lo, hi, s2w)
    return mp.BoundedStateSpace(lo, hi, mp.Euclidean(), mp.OutputMatrix(s2w[1])), orc.StateSpace(lo, hi, s2w)


def _random_segments(n, d, seed, scale=0.3):
    rng = np.random.Generator(np.random.PCG64(seed))
    V = rng.random((n, d)) * 1.1 - 0.05          # a few states out of bounds on purpose
    W = V + (rng.random((n, d)) - 0.5) * scale
    return V, W


@pytest.mark.parametrize("name", list(fx.ALL_2D))
@pytest.mark.parametrize("fixed", [False, True])
def test_k6_k7_2d_fixture_sets(gpu, orc, name, fixed):
    mp = gpu
    spec = fx.ALL_2D[name]
    CC = mp.PointRobot2D(fx.product_shape(mp, spec), fixed_point_test=fixed)
    O = orc.Obstacles2D(spec, fixed_point_test=fixed)
    SSp, SSo = _space_pair(mp, orc, [0, 0], [1, 1])
    V, W = _random_segments(200_000, 2, 1234)
    assert np.array_equal(mp.states_free(V, CC, SSp), orc.states_free(O, SSo, V))
    got = mp.segments_free(V, W, CC, SSp)
    exp, cnt = orc.motions_free_straight(O, SSo, V[:20000], W[:20000])
    assert np.array_equal(got[:20000], exp)
    # full size against the workspace-level oracle batch (in-bounds starts only)
    inb = np.all((V >= 0) & (V <= 1), axis=1)
    assert np.array_equal(got[inb], O.segments_free(V[inb], W[inb]))
    assert not got[~inb].any()
    if name != "EMPTY_2D":
        assert 0.02 < (~got[inb]).mean() < 0.98


def test_k7_nested_compound_and_degenerate_segments(gpu, orc):
    mp = gpu
    inner = ("compound", [("circle", (0.2, 0.2), 0.05), fx.box2d([0.6, 0.7], [0.6, 0.7])])
    spec = ("compound", [inner, ("circle", (0.8, 0.2), 0.05), ("compound", [])])
    CC = mp.PointRobot2D(fx.product_shape(mp, spec))
    O = orc.Obstacles2D(spec)
    V, W = _random_segments(50_000, 2, 77, scale=0.8)
    W[:1000] = V[:1000]                                   # zero-length segments
    W[1000:2000, 0] = V[1000:2000, 0]                     # vertical
    W[2000:3000, 1] = V[2000:3000, 1]                     # horizontal
    assert np.array_equal(mp.segments_free(V, W, CC), O.segments_free(V, W))
    assert np.array_equal(mp.states_free(V, CC), O.points_free(V))
    # addobstacle / addblocker nest exactly like the reference (robots2D.jl:23-24)
    CC2 = mp.addblocker(mp.addobstacle(CC, mp.Box2D([0.4, 0.5], [0.1, 0.2])), [0.5, 0.9], 0.07)
    O2 = orc.Obstacles2D(("compound", [("compound", [spec, fx.box2d([0.4, 0.5], [0.1, 0.2])]), ("circle", (0.5, 0.9), 0.07)]))
    assert np.array_equal(mp.segments_free(V, W, CC2), O2.segments_free(V, W))


@pytest.mark.parametrize("d,boxes", [(2, "BOXES2D"), (3, "BOXES3D"), (10, "RANDOM10")])
def test_k6_k8_boxes(gpu, orc, d, boxes):
    mp = gpu
    bl = fx.random_hyperboxes(64, 10, 20240613) if boxes == "RANDOM10" else getattr(fx, boxes)
    CC = mp.PointRobotNDBoxes([mp.BoxBounds(*b) if isinstance(b, tuple) else mp.BoxBounds(b) for b in bl])
    B = orc.Boxes(bl)
    lo, hi = np.zeros(d), np.ones(d)
    SSp, SSo = _space_pair(mp, orc, lo, hi)
    V, W = _random_segments(100_000, d, 99 + d, scale=0.5 if d < 10 else 1.6)
    W[:500] = V[:500]
    W[500:1500, 0] = V[500:1500, 0]                       # zero components: IEEE division by zero (Q2)
    assert np.array_equal(mp.states_free(V, CC, SSp), orc.states_free(B, SSo, V))
    got = mp.segments_free(V, W, CC, SSp)
    inb = np.all((V >= 0) & (V <= 1), axis=1)
    assert np.array_equal(got[inb], B.segments_free(V[inb], W[inb]))
    assert not got[~inb].any()
    exp, _ = orc.motions_free_straight(B, SSo, V[:5000], W[:5000])
    assert np.array_equal(got[:5000], exp)
    assert 0 < (~got[inb]).mean() < 0.98


def test_k6_k8_double_integrator_workspace_maps(gpu, orc):
    mp = gpu
    CCb = mp.PointRobotNDBoxes([mp.BoxBounds(b) for b in fx.BOXES2D])
    CCs = mp.PointRobot2D(fx.product_shape(mp, fx.ISRR_2H))
    B, O = orc.Boxes(fx.BOXES2D), orc.Obstacles2D(fx.ISRR_2H)
    lo, hi = [0, 0, -1.5, -1.5], [1, 1, 1.5, 1.5]
    rng = np.random.Generator(np.random.PCG64(5))
    V = rng.random((50_000, 4)) * [1.1, 1.1, 3.2, 3.2] - [0.05, 0.05, 1.6, 1.6]
    W = V + (rng.random((50_000, 4)) - 0.5) * 0.4
    C = np.hstack([np.eye(2), np.zeros((2, 2))])
    for s2w in (("matrix", C), ("view", [1, 2])):
        SSp, SSo = _space_pair(mp, orc, lo, hi, s2w)
        for CC, R in ((CCb, B), (CCs, O)):
            assert np.array_equal(mp.states_free(V, CC, SSp), orc.states_free(R, SSo, V))
            exp, _ = orc.motions_free_straight(R, SSo, V[:8000], W[:8000])
            assert np.array_equal(mp.segments_free(V[:8000], W[:8000], CC, SSp), exp)


def _check_table(orc, V, r, D, q0=0, q1=None):
    ref = orc.KDTree(V).rball(r, q0, q1 if q1 is not None else len(V))
    assert np.array_equal(D.colptr, ref[0])
    assert np.array_equal(D.rowval, ref[1])
    assert D.nzval.tobytes() == ref[2].tobytes()           # distances bit-identical
    return ref


@pytest.mark.parametrize("d,N,r", [(2, 1000, None), (2, 50_000, None), (3, 20_000, 0.06), (2, 3000, 0.0), (2, 7, 0.5)])
def test_k1_k2_rball_matches_oracle(gpu, orc, d, N, r):
    mp = gpu
    V = fx.uniform_samples(N, d, 20240601 + N)
    if r is None:
        r = fx.fmt_radius(N, d)
    NN = mp.MetricNN(V)
    cache = NN.precompute(r)
    ref = _check_table(orc, V, r, cache.D)
    if N <= 3000:                                          # the brute-force truth as well
        b = orc.rball_brute(V, r)
        assert np.array_equal(b[1], cache.D.rowval)
    # column views (nearneighbors.jl:128) and filtered views (:104-107)
    v = N // 2 + 1
    col = mp.inball(NN, v, r)
    assert np.array_equal(col.nzind, ref[1][ref[0][v - 1] - 1:ref[0][v] - 1])
    f = np.zeros(N, dtype=bool)
    f[::2] = True
    fcol = mp.inballB(NN, v, r, f)
    assert np.array_equal(fcol.nzind, col.nzind[f[col.nzind - 1]])
    NN.close()


@pytest.mark.parametrize("d,N", [(4, 4000), (6, 3000), (10, 5000), (16, 1500), (1, 2000)])
def test_k3_k4_high_dim_rball_matches_oracle(gpu, orc, d, N):
    """all-pairs FP32 prefilter + exact FP64 recheck: same sets, bit-identical distances"""
    mp = gpu
    V = fx.uniform_samples(N, d, 20240603 + d)
    r = fx.fmt_radius(N, d) if d > 1 else 0.01
    NN = mp.MetricNN(V)
    D = NN.precompute(r).D
    ref = orc.rball_brute(V, r)
    assert np.array_equal(D.colptr, ref[0]) and np.array_equal(D.rowval, ref[1])
    assert D.nzval.tobytes() == ref[2].tobytes()
    assert D.nnz > N
    NN.close()


def test_k3_prefilter_band_has_no_false_negatives(gpu, orc):
    """adversarial for the FP32 CUDA-core prefilter: pairs EXACTLY at the radius, large coordinate offsets
    (FP32 conversion error >> the gap to the radius), shard ranges.  The cloud is wide against r (2 delta / r^2
    ~ 0.8 - 1), so the build takes the CUDA-core sweep, not the tensor cores; the tensor-core form of this test is
    the c-band cases of test_gpu_k3_paths.py."""
    mp = gpu
    rng = np.random.Generator(np.random.PCG64(17))
    d = 5
    base = rng.integers(-40, 40, size=(600, d)).astype(np.float64)
    V = np.vstack([base, base + [3, 4, 0, 0, 0], base + [0, 0, 5, 0, 0], base + [3, 0, 4, 0, 1e-9]]) / 8.0
    for off, r in ((0.0, 5.0 / 8.0), (1000.0, 5.0 / 8.0), (-3.0e4, 0.7)):
        W = V + off
        NN = mp.MetricNN(W)
        NN.set_query_range(100, 1900)
        D = NN.precompute(r).D
        ref = orc.rball_brute(W, r, 0, 100, 1900)
        assert np.array_equal(D.colptr, ref[0]) and np.array_equal(D.rowval, ref[1])
        assert D.nzval.tobytes() == ref[2].tobytes()
        if r == 5.0 / 8.0:
            assert (D.nzval == r).sum() > 500        # the exactly-at-radius pairs are members
        NN.close()


def test_k2_duplicates_clusters_and_big_columns(gpu, orc):
    """ragged inputs: coincident points, a dense cluster whose columns exceed the per-warp stage
    (spill path), points outside the unit square, an isolated point"""
    mp = gpu
    rng = np.random.Generator(np.random.PCG64(3))
    V = np.vstack([rng.random((4000, 2)),
                   0.5 + 0.004 * rng.random((600, 2)),      # 600 points within one r-ball
                   rng.random((50, 2))[[0] * 20],           # 20 exact duplicates
                   np.array([[5.0, -3.0], [0.2, 0.2], [0.2, 0.2]])])
    r = 0.02
    NN = mp.MetricNN(V)
    D = NN.precompute(r).D
    _check_table(orc, V, r, D)
    deg = np.diff(D.colptr)
    assert deg.max() >= 599 and deg.min() == 0
    NN.close()


def test_k2_query_range_shards_concatenate(gpu, orc):
    mp = gpu
    V = fx.uniform_samples(30_000, 2, 8)
    r = fx.fmt_radius(30_000, 2)
    full = orc.KDTree(V).rball(r)
    parts = []
    for q0, q1 in ((0, 10_000), (10_000, 10_001), (10_001, 30_000)):
        NN = mp.MetricNN(V)
        NN.set_query_range(q0, q1)
        D = NN.precompute(r).D
        _check_table(orc, V, r, D, q0, q1)
        parts.append((D.colptr.copy(), D.rowval.copy(), D.nzval.copy()))
        NN.close()
    assert np.array_equal(np.concatenate([p[1] for p in parts]), full[1])


def test_edges_and_points_over_table(gpu, orc):
    """config C1-like: N=1000 in the unit square, ISRR_2H through both checkers"""
    mp = gpu
    N = 1000
    V = fx.uniform_samples(N, 2, 20240601)
    V[0] = [0.1, 0.1]
    V[-1] = [0.9, 0.9]
    r = fx.fmt_radius(N, 2)
    SSp, SSo = _space_pair(mp, orc, [0, 0], [1, 1])
    for CC, R in ((mp.PointRobot2D(mp.obstaclesets.ISRR_2H()), orc.Obstacles2D(fx.ISRR_2H)),
                  (mp.PointRobotNDBoxes([mp.BoxBounds(b) for b in fx.BOXES2D]), orc.Boxes(fx.BOXES2D))):
        NN = mp.MetricNN(V)
        D = NN.precompute(r).D
        F = unpack_bits(NN.points_free(CC, SSp), N)
        assert np.array_equal(F, orc.states_free(R, SSo, V))
        CC.count = 0
        bits, checks = NN.edges_free(NN.table, CC, SSp)
        exp, cnt = orc.edges_free_csc(R, SSo, V, D.colptr, D.rowval)
        assert np.array_equal(unpack_bits(bits, D.nnz), exp.astype(bool))
        assert checks == cnt == CC.count == D.nnz
        # unused high bits of the last chunk are zero (Julia BitVector invariant)
        if D.nnz % 64:
            assert int(bits[-1]) >> (D.nnz % 64) == 0
        NN.close()


def test_full_size_c2_properties(gpu, orc):
    """BASELINE config 2 at full size (N = 1M): oracle kd-tree parity on the whole table plus
    size-independent properties (symmetry, sortedness, validity symmetric under the 2-D SAT
    for in-bounds samples is NOT assumed -- only checked against the oracle on a sample)."""
    mp = gpu
    N = 1_000_000
    V = fx.uniform_samples(N, 2, 20240602)
    r = fx.fmt_radius(N, 2)
    NN = mp.MetricNN(V)
    D = NN.precompute(r).D
    deg = np.diff(D.colptr)
    assert abs(deg.mean() - 2 * np.log(N)) < 0.5
    cols = np.repeat(np.arange(1, N + 1, dtype=np.int64), deg)
    assert not (D.rowval == cols).any()
    # ascending rows inside every column
    d = np.diff(D.rowval)
    starts = D.colptr[1:-1] - 1
    ok = d > 0
    ok[starts[(starts > 0) & (starts < len(D.rowval))] - 1] = True
    assert ok.all()
    # symmetric relation with identical distances: sort (i,j) and (j,i) keys
    k1 = cols * (N + 1) + D.rowval
    k2 = D.rowval * (N + 1) + cols
    o1, o2 = np.argsort(k1, kind="stable"), np.argsort(k2, kind="stable")
    assert np.array_equal(k1[o1], k2[o2]) and np.array_equal(D.nzval[o1], D.nzval[o2])
    assert (D.nzval <= r).all() and (D.nzval * D.nzval <= r * r * (1 + 1e-15)).all()
    # oracle on a 20k-column slice (the kd-tree oracle does 1M columns in ~seconds, but keep it short)
    ref = orc.KDTree(V).rball(r, 500_000, 520_000)
    lo, hi = D.colptr[500_000] - 1, D.colptr[520_000] - 1
    assert np.array_equal(D.rowval[lo:hi], ref[1]) and D.nzval[lo:hi].tobytes() == ref[2].tobytes()
    # edges: all 27.6M bits vs the oracle on the same slice
    CC = mp.PointRobot2D(mp.obstaclesets.ISRR_2H())
    SSp, SSo = _space_pair(mp, orc, [0, 0], [1, 1])
    bits, checks = NN.edges_free(NN.table, CC, SSp)
    assert checks == D.nnz
    got = unpack_bits(bits, D.nnz)
    exp, _ = orc.edges_free_csc(orc.Obstacles2D(fx.ISRR_2H), SSo, V, ref[0], ref[1], 500_000)
    assert np.array_equal(got[lo:hi], exp.astype(bool))
    NN.close()


@pytest.mark.parametrize("checker", ["sat2d", "sat2d_nested", "boxes2d", "boxes3d"])
def test_fused_build_checked_equals_separate_calls(gpu, orc, checker):
    """mpb200_inball_build_checked (K2 with K7/K8 fused) == inball_build + edges_free == oracle,
    including columns that overflow the thread path (dense cluster -> big-column leftovers)"""
    mp = gpu
    rng = np.random.Generator(np.random.PCG64(99))
    d = 3 if checker == "boxes3d" else 2
    N = 60_000
    V = rng.random((N, d)) * 1.04 - 0.02                      # some samples outside the unit cube
    V[:300] = 0.3 + 0.002 * rng.random((300, d))              # cluster: columns with ~300 entries
    r = fx.fmt_radius(N, d)
    lo, hi = np.zeros(d), np.ones(d)
    SSp, SSo = _space_pair(mp, orc, lo, hi)
    if checker == "sat2d":
        CC, R = mp.PointRobot2D(mp.obstaclesets.ISRR_POLY_WITH_SPIKE()), orc.Obstacles2D(fx.ISRR_POLY_WITH_SPIKE)
    elif checker == "sat2d_nested":
        spec = ("compound", [fx.TRI_BALLS, ("circle", (0.8, 0.8), 0.1), fx.box2d([0.05, 0.2], [0.7, 0.9])])
        CC, R = mp.PointRobot2D(fx.product_shape(mp, spec)), orc.Obstacles2D(spec)
    elif checker == "boxes2d":
        CC, R = mp.PointRobotNDBoxes([mp.BoxBounds(b) for b in fx.BOXES2D]), orc.Boxes(fx.BOXES2D)
    else:
        CC, R = mp.PointRobotNDBoxes([mp.BoxBounds(b) for b in fx.BOXES3D]), orc.Boxes(fx.BOXES3D)
    NN = mp.MetricNN(V)
    CC.count = 0
    cache, bits, checks = NN.precompute_checked(r, CC, SSp)
    D = cache.D
    ref = _check_table(orc, V, r, D)
    exp, cnt = orc.edges_free_csc(R, SSo, V, D.colptr, D.rowval)
    got = unpack_bits(bits, D.nnz)
    assert np.array_equal(got, exp.astype(bool))
    assert checks == cnt == CC.count
    assert np.diff(D.colptr).max() >= 299
    # and the stand-alone edge kernel on the same table
    bits2, checks2 = NN.edges_free(NN.table, CC, SSp)
    assert np.array_equal(unpack_bits(bits2, D.nnz), got) and checks2 == cnt
    if D.nnz % 64:
        assert int(bits[-1]) >> (D.nnz % 64) == 0
    NN.close()


def test_k3_single_sweep_slab_overflow_falls_back(gpu, orc):
    """the slab capacity is sized from a probe of the first 2048 columns; a dense cluster among
    later indices overflows it and the build must fall back to the two-sweep fill.  The cluster far away makes
    the cloud wide against r (2 delta / r^2 ~ 2.3), so this exercises the FP32 CUDA-core sweep; overflow after a
    tensor-core sweep is the d-overflow cases of test_gpu_k3_paths.py."""
    mp = gpu
    rng = np.random.Generator(np.random.PCG64(5))
    d = 5
    V = np.vstack([rng.random((3000, d)), 3.0 + 0.01 * rng.random((700, d)), rng.random((300, d))])   # cluster far away
    r = 0.12
    NN = mp.MetricNN(V)
    D = NN.precompute(r).D
    ref = orc.rball_brute(V, r)
    assert np.array_equal(D.colptr, ref[0]) and np.array_equal(D.rowval, ref[1])
    assert D.nzval.tobytes() == ref[2].tobytes()
    deg = np.diff(D.colptr)
    assert deg[:2048].max() * 1.5 + 64 < deg.max()        # the probe really underestimates
    NN.close()


@pytest.mark.parametrize("d", [2, 3])
def test_k2_stripe_sorted_shards_use_restricted_grid(gpu, orc, d):
    """samples stored in stripe order: every shard's query range is a spatial stripe, its grid only
    covers the stripe + r, and out-of-stripe samples are never inserted -- results unchanged"""
    mp = gpu
    N = 40_000
    V = fx.uniform_samples(N, d, 31 + d)
    V = V[np.argsort(V[:, 0], kind="stable")]
    r = fx.fmt_radius(N, d) * 1.3
    full = orc.KDTree(V).rball(r)
    got_rows, got_vals = [], []
    CC = mp.PointRobotNDBoxes([mp.BoxBounds(b) for b in (fx.BOXES2D if d == 2 else fx.BOXES3D)])
    SSp, SSo = _space_pair(mp, orc, np.zeros(d), np.ones(d))
    B = orc.Boxes(fx.BOXES2D if d == 2 else fx.BOXES3D)
    for q0, q1 in ((0, 9_000), (9_000, 9_001), (9_001, 31_000), (31_000, N)):
        NN = mp.MetricNN(V)
        NN.set_query_range(q0, q1)
        cache, bits, checks = NN.precompute_checked(r, CC, SSp)
        ref = orc.KDTree(V).rball(r, q0, q1)
        assert np.array_equal(cache.D.colptr, ref[0]) and np.array_equal(cache.D.rowval, ref[1])
        assert cache.D.nzval.tobytes() == ref[2].tobytes()
        exp, cnt = orc.edges_free_csc(B, SSo, V, ref[0], ref[1], q0)
        assert np.array_equal(unpack_bits(bits, cache.D.nnz), exp.astype(bool)) and checks == cnt
        F = unpack_bits(NN.points_free(CC, SSp), q1 - q0)
        assert np.array_equal(F, orc.states_free(B, SSo, V[q0:q1]))
        got_rows.append(cache.D.rowval.copy())
        NN.close()
    assert np.array_equal(np.concatenate(got_rows), full[1])


@pytest.mark.parametrize("d", [2, 3])
def test_k6_cell_ordered_points_equal_index_ordered(gpu, orc, d):
    """points_free walks the samples in grid-cell order once a grid exists (and over a shard's own range):
    same bits as the index-ordered pass before any build, and as the oracle."""
    mp = gpu
    N = 30_011   # not a multiple of 32 or 64
    V = fx.uniform_samples(N, d, 77) * 1.06 - 0.03   # some points out of bounds
    SSp, SSo = _space_pair(mp, orc, [0] * d, [1] * d)
    if d == 2:
        CC, R = mp.PointRobot2D(mp.obstaclesets.ISRR_2H()), orc.Obstacles2D(fx.ISRR_2H)
    else:
        CC, R = mp.PointRobotNDBoxes([mp.BoxBounds(b) for b in fx.BOXES3D]), orc.Boxes(fx.BOXES3D)
    exp = orc.states_free(R, SSo, V)
    NN = mp.MetricNN(V)
    before = unpack_bits(NN.points_free(CC, SSp), N).copy()
    NN.build_table(0.02 if d == 2 else 0.05)
    after = unpack_bits(NN.points_free(CC, SSp), N).copy()
    assert np.array_equal(before, exp) and np.array_equal(after, exp)
    q0, q1 = 10_007, 20_033
    NN.set_query_range(q0, q1)
    shard_before = unpack_bits(NN.points_free(CC, SSp), q1 - q0).copy()
    NN.build_table(0.02 if d == 2 else 0.05)
    shard_after = unpack_bits(NN.points_free(CC, SSp), q1 - q0).copy()
    assert np.array_equal(shard_before, exp[q0:q1]) and np.array_equal(shard_after, exp[q0:q1])
    NN.close()
