"""Small end-to-end exercise of every kernel family, for compute-sanitizer (memcheck / racecheck / initcheck)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import mpb200
mpb200.init(0)
rng = np.random.Generator(np.random.PCG64(1))
SS = mpb200.UnitHypercube(2)
CC = mpb200.PointRobot2D(mpb200.obstaclesets.ISRR_2H(), fixed_point_test=True)
# grid r-ball (d = 2, 3), incl. shard mode, big columns, cell-ordered validity passes
for d, N, r in ((2, 6000, 0.03), (3, 3000, 0.12)):
    V = rng.random((N, d))
    NN = mpb200.MetricNN(V)
    NN.precompute(r)
    if d == 2:
        NN.points_free(CC, SS); NN.edges_free(NN.table, CC, SS)
        NN.set_query_range(1000, 4000); NN.build_table(r); NN.points_free(CC, SS); NN.edges_free(NN.table, CC, SS)
    NN.close()
V = rng.random((500, 2)) * 0.05
NN = mpb200.MetricNN(V); NN.precompute(1.0); NN.edges_free(NN.table, CC, SS); NN.close()       # big-column path
# x-sorted shard
V = rng.random((8000, 2)); V = V[np.argsort(V[:, 0])]
NN = mpb200.MetricNN(V); NN.set_query_range(2000, 5000); NN.precompute(0.03); NN.close()
# d >= 4: tensor-core prefilter + CUDA-core fallback dimension
for d in (6, 16):
    V = rng.random((1500, d)); NN = mpb200.MetricNN(V); NN.precompute(0.9 if d == 6 else 1.4); NN.close()
# d >= 4 shard with unaligned ends (one-sided tensor-core sweep, estimated cap), and 500 samples pairwise farther
# apart than r (empty probe: cap = 0, the count-only sweep decides colptr)
V = rng.random((3000, 6)); NN = mpb200.MetricNN(V); NN.set_query_range(37, 2461); NN.precompute(0.6); NN.close()
idx = rng.choice(3 ** 6, size=500, replace=False)
V = ((idx[:, None] // 3 ** np.arange(6)) % 3) * 0.5; NN = mpb200.MetricNN(V); NN.precompute(0.45); NN.close()
# boxes
B = mpb200.PointRobotNDBoxes([mpb200.BoxBounds(np.array([[0.2, 0.4], [0.2, 0.4], [0.0, 1.0]]))])
V = rng.random((3000, 3)); NN = mpb200.MetricNN(V); NN.precompute(0.1)
NN.points_free(B, mpb200.UnitHypercube(3)); NN.edges_free(NN.table, B, mpb200.UnitHypercube(3)); NN.close()
# LQ
DI = mpb200.DoubleIntegrator(2)
V = np.hstack([rng.random((800, 2)), rng.random((800, 2)) * 2 - 1])
Q = mpb200.QuasiMetricNN(V, DI.dist); Q.precompute(0.8); Q.lq_edges_free(CC, DI); Q.close()
# sampling (both orders) and Monte Carlo
mpb200.MetricNN.sample_free(CC, SS, 5000, seed=1).close()
mpb200.MetricNN.sample_free(CC, SS, 5000, seed=1, order="morton").close()
Bx = mpb200.PointRobotNDBoxes([mpb200.BoxBounds(np.array([0.5, -10.0]), np.array([10.0, 10.0]))])
P = mpb200.MCProblem(np.eye(2)[None], (np.eye(2) * 0.1)[None], np.eye(2), np.array([[0.2, 0.0]] * 2), [0.3, 0.7], [[3.0, 0.0]])
mpb200.collision_probability(P, Bx, 20000, seed=3)
# round 2: general linear-affine LQ (numeric 2BVP), batched closest / closeR, pipe peaks, table write floor,
# the narrowed table fetch, and the peer exchange in a world of one (pack kernel + flag barrier on the own buffer)
import ctypes
from mpb200 import _lib, sharding
A = np.array([[0.0, 1.0, 0.0], [0.0, 0.0, 1.0], [0.0, 0.0, 0.0]]); Bm = np.array([[0.0], [0.0], [1.0]])
LQ = mpb200.linearquadratic.LinearQuadraticQuasiMetricSpace(np.array([0, -1.0, -2.0]), np.array([1, 1.0, 2.0]), A, Bm,
                                                            np.array([0.0, 0.1, 0.2]), np.array([[2.0]]),
                                                            np.array([[1.0, 0, 0], [0, 1.0, 0]]))
V = np.array([0, -1.0, -2.0]) + rng.random((400, 3)) * np.array([1, 2.0, 4.0])
Q = mpb200.QuasiMetricNN(V, LQ.dist); Q.precompute(1.3); Q.lq_edges_free(CC, LQ)
mpb200.linearquadratic.lq_motions_free(V[:50], V[50:100], CC, LQ, 1.3); Q.close()
Wm = np.tile(np.array([[2.0, 0.3], [0.3, 1.0]]), (300, 1, 1))
mpb200.montecarlo.close_points(rng.random((300, 2)), CC, Wm, 0.2, want_all=True)
B4 = mpb200.PointRobotNDBoxes([mpb200.BoxBounds(np.full(4, 0.2), np.full(4, 0.5)), mpb200.BoxBounds(np.full(4, 0.6), np.full(4, 0.9))])
mpb200.montecarlo.close_points(rng.random((100, 4)), B4, np.tile(np.eye(4) + 0.1, (100, 1, 1)), 1.0)
lib = mpb200.load()
v = ctypes.c_double(0.0)
for kind in (0, 1, 2):
    _lib.check(lib.mpb200_pipe_peak(kind, ctypes.byref(v)))
V = rng.random((60000, 2)); NN = mpb200.MetricNN(V); NN.precompute(0.02)          # > 2^20 entries: narrowed fetch
_lib.check(lib.mpb200_table_write_floor(NN.table.h, ctypes.byref(v)))
NN.edges_free(NN.table, CC, SS, fetch=False, count=False)
x = _lib.c_vp(); h = (ctypes.c_char * 64)()
_lib.check(lib.mpb200_xchg_create(0, 1, 60000, (NN.table.nnz + 63) // 64 + 1, ctypes.byref(x), h))
_lib.check(lib.mpb200_xchg_connect(x, h)); _lib.check(lib.mpb200_xchg_attach(x, NN.table.h))
for _ in range(2):
    NN.build_table(0.02); NN.edges_free(NN.table, CC, SS, fetch=False, count=False); _lib.check(lib.mpb200_xchg_push(x, NN.table.h))
st = _lib.c_i64(0)
_lib.check(lib.mpb200_xchg_view(x, None, None, None, None, ctypes.byref(st))); assert st.value == 0
_lib.check(lib.mpb200_xchg_attach(None, NN.table.h)); _lib.check(lib.mpb200_xchg_destroy(x)); NN.close()
# later in round 2: car spaces (steer, chopped tables both kinds, sharded range, edge + motion checks, both obstacle
# kinds) and k-nearest connections (k-selection, mutual neighbourhoods)
Vc = np.column_stack([rng.random(700), rng.random(700), rng.uniform(0, 2 * np.pi, 700)])
Bc = mpb200.PointRobotNDBoxes([mpb200.BoxBounds(np.array([0.3, 0.3]), np.array([0.5, 0.6]))])
for mk, cls in ((mpb200.ReedsSheppMetricSpace, mpb200.MetricNN), (mpb200.DubinsQuasiMetricSpace, mpb200.QuasiMetricNN)):
    S3 = mk(0.05, 0.9)
    mpb200.setup_steering(S3, 0.2)
    Nc = cls(Vc, S3.dist, Vc[0]); Nc.precompute(0.2); Nc.car_edges_free(CC, S3); Nc.car_edges_free(Bc, S3)
    Nc.set_query_range(100, 500); Nc.precompute(0.2); Nc.car_edges_free(CC, S3)
    mpb200.car_steer_batch(S3, Vc[:64], Vc[64:128]); mpb200.car_motions_free(Vc[:64], Vc[64:128], CC, S3); Nc.close()
Vk = rng.random((3000, 2)); Nk = mpb200.MetricNN(Vk); Nk.precompute_knn(12); Nk.edges_free(Nk.table_knn, CC, SS); Nk.close()
Vk = rng.random((900, 6)); Nk = mpb200.MetricNN(Vk); Nk.precompute_knn(9); Nk.close()
print("sanitize run complete")
