/*
 * mpb200.h -- C ABI of libmpb200.so, the B200 (sm_100a) back-end for the
 * data-parallel hot path of schmrlng/MotionPlanning.jl.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types.
 * A Julia maintainer binds these with `ccall((:sym, "libmpb200"), Cint, ...)`
 * (see INTEGRATION.md and julia/MotionPlanningB200.jl); the Python host mirror
 * in motionplanning.jl_b200/ binds them with ctypes.
 *
 * Conventions
 *  - every function returns 0 on success, a negative MPB200_E* code otherwise;
 *    mpb200_last_error() returns the thread-local message.  No CPU fallback:
 *    without a usable sm_100 GPU every compute entry point fails.
 *  - host buffers are caller-owned (Julia GC / numpy); the library copies inputs
 *    at *_create and writes outputs only between call and return.  Calls that hand
 *    data back wait for it; calls whose result pointers are all NULL only enqueue
 *    work on the launching stream (noted at each entry point).
 *  - samples cross as the reference stores them: Vector{SVector{d,Float64}} ==
 *    column-major d x N Float64 (primitivetypes.jl:21-23, statevec2mat).
 *  - neighbour tables cross as Julia SparseMatrixCSC{Float64,Int64} fields:
 *    colptr (ncols+1), rowval (nnz, ascending within a column), nzval (nnz),
 *    all indices 1-based Int64 (nearneighbors.jl:23-28, ImmutableNNC.D).
 *  - validity tables cross in Julia BitVector chunk layout: element k (0-based)
 *    is bit (k & 63) of UInt64 word (k >> 6); unused high bits are zero.
 *  - one process drives one GPU (mpb200_init(device)); multi-GPU sharding is by
 *    query (column) range, see mpb200_samples_set_query_range.
 */
#ifndef MPB200_H
#define MPB200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPB200_OK 0
#define MPB200_EARG (-1)    /* bad argument */
#define MPB200_ECUDA (-2)   /* CUDA runtime error / no usable GPU */
#define MPB200_ESTATE (-3)  /* call out of order (e.g. fetch before build) */
#define MPB200_ENOMEM (-4)

typedef struct mpb200_samples mpb200_samples;     /* device copy of a sample set        */
typedef struct mpb200_table mpb200_table;         /* device-resident CSC neighbour table */
typedef struct mpb200_obstacles mpb200_obstacles; /* device copy of an obstacle set      */
typedef struct mpb200_lq mpb200_lq;               /* linear-quadratic 2BVP               */

/* ---- runtime ----------------------------------------------------------- */
/* Select the CUDA device for this process and create the library stream.
 * Fails (MPB200_ECUDA) when there is no GPU or it is not compute capability 10.x. */
int mpb200_init(int device);
void mpb200_shutdown(void);
const char *mpb200_last_error(void);
int mpb200_version(void);
/* Launch on a caller-owned cudaStream_t (e.g. torch's current stream) instead of the
 * library's own; pass NULL to return to the library stream. */
int mpb200_set_stream(void *cuda_stream);
int mpb200_synchronize(void);
/* Device arrays released by the library (destroyed tables / sample sets, outgrown buffers) are parked
 * in a free list and reused by later calls instead of going through cudaFree / cudaMalloc (milliseconds
 * each, device-synchronising).  This returns every parked block to the driver. */
int mpb200_release_cached(void);
/* Pinned host memory for result buffers (fast D2H); plain malloc'ed buffers work too. */
int mpb200_host_alloc(uint64_t bytes, void **out);
int mpb200_host_free(void *p);
/* Number of kernels this library has launched since mpb200_init (bench "gpu_launches"). */
int64_t mpb200_launch_count(void);
/* Device time of the last entry point, milliseconds, measured with CUDA events on the
 * launching stream; phase 0 = whole call, 1.. = entry-point specific (see DESIGN.md).
 * The events are recorded inside the call and read back lazily here (this waits for the
 * recorded work), so entry points that return nothing from the device never block.
 * mpb200_last_ms_of keeps one record per kind of operation, so the three calls of a
 * planning step (table build, point validity, edge validity) can be issued back to back
 * and timed afterwards. */
#define MPB200_OP_TABLE 0  /* mpb200_inball_build / mpb200_lq_inball_build */
#define MPB200_OP_POINTS 1 /* mpb200_points_free */
#define MPB200_OP_EDGES 2  /* mpb200_edges_free / mpb200_lq_edges_free */
#define MPB200_OP_OTHER 3  /* mpb200_mc_collision_probability */
#define MPB200_OP_PLAN 4   /* mpb200_gmt_plan: phase 1 = the planning kernel */
#define MPB200_OP_PATH 5   /* mpb200_shortcut_paths: phase 1 visibility, phase 2 minimum */
double mpb200_last_ms(int phase);
double mpb200_last_ms_of(int op, int phase);

/* ---- sample sets: replaces MetricNN/QuasiMetricNN.V (nearneighbors.jl:62-92) ---- */
int mpb200_samples_create(const double *V_aos, int64_t N, int d, mpb200_samples **out);
int mpb200_samples_destroy(mpb200_samples *s);
/* Restrict this process to query columns [q0, q1) (0-based, half-open) of the table:
 * the multi-GPU shard.  Default is [0, N). */
int mpb200_samples_set_query_range(mpb200_samples *s, int64_t q0, int64_t q1);

/* ---- Euclidean r-ball table --------------------------------------------------
 * Replaces helper_data_structures(V, ::Euclidean) (geometric.jl:14-15: KDTree build)
 * plus inball(V, dist, ::TreeDistanceDS, v, r) for every v in the query range
 * (nearneighbors.jl:179-183), i.e. it produces the ImmutableNNC.D matrix that
 * inball!(NN{..,ImmutableNNC}, v, r) = viewcol(D, v) serves (nearneighbors.jl:128).
 * Member iff j != v and sum_i (V[v]_i - V[j]_i)^2 <= r*r (index order, no FMA);
 * stored value sqrt of the same sum; rows ascending.
 * If *table is non-NULL on entry its device buffers are reused. */
int mpb200_inball_build(mpb200_samples *s, double r, mpb200_table **table, int64_t *nnz);
/* Copy a table to caller buffers; any pointer may be NULL to skip that array.
 * colptr has (q1-q0)+1 entries, relative to the shard (colptr[0] == 1). */
int mpb200_table_fetch(const mpb200_table *t, int64_t *colptr, int64_t *rowval, double *nzval);
int mpb200_table_nnz(const mpb200_table *t, int64_t *nnz, int64_t *ncols);
/* Device pointers of a table's arrays (colptr int64[ncols+1], rowval int64[nnz], nzval f64[nnz],
 * edge_bits uint64[ceil(nnz/64)] = last mpb200_edges_free / mpb200_lq_edges_free result or NULL),
 * valid until the next build on / destroy of the handle: lets the caller hand shards to NCCL
 * (all-gather across the GPUs of a box) without a host round trip. */
int mpb200_table_device_view(const mpb200_table *t, void **colptr, void **rowval, void **nzval, void **edge_bits);
int mpb200_table_destroy(mpb200_table *t);

/* ---- obstacle sets ------------------------------------------------------------ */
/* 2-D compound of circles and convex polygons, PRECOMPUTED on the host exactly as the
 * reference constructors do (SAT2D.jl:12-98): the device never re-derives normals.
 * shape_kind 0 = Circle  (data: cx cy r xlo xhi ylo yhi)
 *            1 = Polygon (data: xlo xhi ylo yhi, K points, K unit normals, K nextrema)
 * gates are the AABBs of enclosing Compound2D nodes (parent index or -1).
 * flags bit0: use the intended point-in-polygon test instead of the reference's
 * inverted one (SAT2D.jl:124-127). */
typedef struct {
    int32_t n_gates;
    const int32_t *gate_parent;
    const double *gate_aabb;
    int32_t n_shapes;
    const int32_t *shape_kind;
    const int32_t *shape_gate;
    const int32_t *shape_off;
    const double *data;
    int32_t flags;
} mpb200_obstacles2d_desc;
/* replaces PointRobot2D(obstacles) (robots2D.jl:5-10) */
int mpb200_obstacles2d_create(const mpb200_obstacles2d_desc *desc, mpb200_obstacles **out);
/* replaces PointRobotNDBoxes(boxes) (boxesND.jl:15-21); lo/hi box-major M x d */
int mpb200_boxes_create(const double *lo, const double *hi, int M, int d, mpb200_obstacles **out);
int mpb200_obstacles_destroy(mpb200_obstacles *o);

/* BoundedStateSpace bounds + State2Workspace (statespaces.jl:29-34,45-60) */
typedef struct {
    int32_t n;           /* state dimension */
    const double *lo;    /* n */
    const double *hi;    /* n */
    int32_t s2w_kind;    /* 0 Identity, 1 VectorView(inds), 2 OutputMatrix(C) */
    int32_t dw;          /* workspace dimension */
    const int32_t *inds; /* dw, 0-based (kind 1) */
    const double *C;     /* dw x n column-major (kind 2) */
} mpb200_space_desc;

/* ---- batched validity ---------------------------------------------------------- */
/* F[i] = is_free_state(V[i], CC, SS) for the samples of the query range [q0, q1) -- all N by
 * default (fmt.jl:31-36, sampling.jl:25; statespaces.jl:151-152; robots2D.jl:12;
 * boxesND.jl:42-43).  bits: ceil((q1-q0)/64) words, bit k = sample q0 + k.
 * bitchunks may be NULL: the call then only enqueues the work (no wait); the bits stay on the
 * device, ordered on the launching stream before every later call. */
int mpb200_points_free(const mpb200_samples *s, const mpb200_obstacles *o, const mpb200_space_desc *ss,
                       uint64_t *bitchunks);
/* For every stored entry (row y, column x) of a table, in storage order:
 * is_free_motion(V[y], V[x], CC, SS) with straight-line waypoints (fmt.jl:75;
 * statespaces.jl:153-158; geometric.jl:20; robots2D.jl:13-14; boxesND.jl:52-56).
 * bits: ceil(nnz/64) words.  *checks receives the number of segment checks that
 * CC.count would have been incremented by.  With bitchunks == NULL and checks == NULL the call
 * only enqueues the work (no wait); read the bits later with mpb200_table_fetch_edge_bits. */
int mpb200_edges_free(const mpb200_samples *s, const mpb200_table *t, const mpb200_obstacles *o,
                      const mpb200_space_desc *ss, uint64_t *bitchunks, int64_t *checks);
/* Convenience for config "batched r-ball neighbours + edge validity precompute": build the
 * Euclidean r-ball table and the validity of every stored edge with one call (= mpb200_inball_build
 * followed by mpb200_edges_free); the edge bits stay on the device with the table
 * (mpb200_table_fetch_edge_bits / mpb200_table_device_view). */
int mpb200_inball_build_checked(mpb200_samples *s, double r, const mpb200_obstacles *o, const mpb200_space_desc *ss,
                                mpb200_table **table, int64_t *nnz, int64_t *checks);
int mpb200_table_fetch_edge_bits(const mpb200_table *t, uint64_t *bitchunks);
/* State-level batches for callers that hold states, not indices (sampling.jl:25,
 * postprocessors.jl:11,21): n states / n straight segments, AoS d x n; out: 1 byte each. */
int mpb200_states_free(const double *v_aos, int64_t n, int d, const mpb200_obstacles *o,
                       const mpb200_space_desc *ss, uint8_t *out);
int mpb200_segments_free(const double *v_aos, const double *w_aos, int64_t n, int d, const mpb200_obstacles *o,
                         const mpb200_space_desc *ss, uint8_t *out);

/* Batched sample_free!(P, N) (sampling.jl:23-37; SURVEY 8(f).1): draws states uniformly in the state bounds
 * (sample_space, statespaces.jl) and keeps the first N for which is_free_state(v, CC, SS) holds -- generated,
 * tested and compacted on the device, so the sample set never crosses PCIe on its way in.  The reference draws
 * from Julia's global RNG, which cannot be reproduced; the candidate stream here is specified in
 * oracle/sample.c (Philox4x32-10 keyed by seed, counter = candidate number) and is independent of launch
 * geometry: the same (obstacles, space, N, seed) always yields the same samples, in candidate order.
 * order = MPB200_ORDER_MORTON numbers the accepted samples along a Z-order curve over the first min(n, 3)
 * coordinates (stable: ties keep candidate order) instead of in the order they were drawn: FMT* does not care how
 * i.i.d. samples are numbered, and with a spatially coherent numbering the neighbour-table and validity kernels
 * run about 12% faster (their column writes and gathers become local).
 * V_host (N x n, may be NULL) receives a host copy; *candidates the number of candidates consumed. */
#define MPB200_ORDER_CANDIDATE 0
#define MPB200_ORDER_MORTON 1
int mpb200_sample_free(const mpb200_obstacles *o, const mpb200_space_desc *ss, int64_t N, uint64_t seed, int32_t order,
                       mpb200_samples **out, double *V_host, int64_t *candidates);

/* ---- linear-quadratic steering cost ("ControlNN") --------------------------------
 * Replaces LinearQuadratic(A, B, c, R) / LinearQuadratic2BVP (linearquadratic.jl:6-39,126-157) for
 * xdot = A x + B u + c, cost int (1 + u'Ru).  A (n x n), B (n x m), R (m x m) column-major, c (n); n, m <= 6.
 * As in the reference, A must be nilpotent (expAt, :94-98); R symmetric positive definite; (A, B)
 * controllable.  Two evaluation paths, chosen here:
 *   - the DoubleIntegrator family (:46-53: n = 2m, A = [0 I; 0 0], B = [0; I], c = 0, m = 1..3) uses the
 *     closed form cost(t) = t + alpha/t^3 - beta/t^2 + gamma/t (csrc/lq.cu);
 *   - every other system (drift c != 0, integrator chains, general B) evaluates G(t), xbar(t) and the
 *     cost derivatives numerically from per-system tables (csrc/lq_general.cu; spec in oracle/lq_general.c,
 *     pinned to the reference's SymPy construction by tests/golden/lq_general.json).
 * Anything the reference rejects returns MPB200_EARG with the reference's message. */
int mpb200_lq_create(const double *A, const double *B, const double *c, const double *R, int n, int m,
                     mpb200_lq **out);
int mpb200_lq_destroy(mpb200_lq *lq);
/* Replaces helper_data_structures(V, ::LinearQuadratic) (linearquadratic.jl:68-77): the batched
 * steer_pairwise (:196-225: dcost(r) > 0 prefilter, safeguarded Newton :175-190, cost <= r)
 * plus the inball filter (nearneighbors.jl:165-177), for every column of the query range.
 * tableF column v: { j != v : cost(V[v] -> V[j]) <= r }  (DSF = Dmat', served by inballF!)
 * tableB column v: { j != v : cost(V[j] -> V[v]) <= r }  (DSB = Dmat , served by inballB!)
 * stored value = the cost; rows ascending.  Non-NULL *table handles are reused. */
int mpb200_lq_inball_build(mpb200_samples *s, const mpb200_lq *lq, double r, mpb200_table **tableF,
                           mpb200_table **tableB, int64_t *nnzF, int64_t *nnzB);
/* steer(L, v, w, r) = (cost, t*) for n explicit pairs (linearquadratic.jl:191-195); AoS 2m x n */
int mpb200_lq_steer(const mpb200_lq *lq, const double *v_aos, const double *w_aos, int64_t n, double r,
                    double *cost, double *topt);
/* is_free_motion(V[y], V[x], CC, SS) for every stored entry (row y, column x) of a table, with
 * collision_waypoints(::LinearQuadratic) = 5 states along the optimal trajectory
 * (linearquadratic.jl:85-88; statespaces.jl:153-158).  bits/checks as mpb200_edges_free. */
int mpb200_lq_edges_free(const mpb200_samples *s, const mpb200_table *t, const mpb200_lq *lq, double r,
                         const mpb200_obstacles *o, const mpb200_space_desc *ss, uint64_t *bitchunks,
                         int64_t *checks);
/* the same for n explicit state pairs (fmt.jl:75 called with states) */
int mpb200_lq_motions_free(const mpb200_lq *lq, double r, const double *v_aos, const double *w_aos, int64_t n,
                           const mpb200_obstacles *o, const mpb200_space_desc *ss, uint8_t *out, int64_t *checks);

/* ---- chopped-metric car spaces (Dubins / Reeds-Shepp) --------------------------------------------
 * Replaces, for SE2 states (x, y, theta; AoS 3 x N):
 *   ReedsSheppExact / DubinsExact and their evaluate = reedsshepp / dubins (simplecars.jl:5-27, 196-213, 266-364),
 *   ChoppedMetric / ChoppedQuasiMetric evaluation (primitivetypes.jl:79-100),
 *   helper_data_structures(V, ::Chopped...{ReedsSheppExact|DubinsExact}) = KD-tree over (x, y) (simplecars.jl:42-52)
 *   + inball(V, ::ChoppedPreMetric, ::TreeDistanceDS, v, r, forwards) (nearneighbors.jl:185-198),
 *   steering_control / propagate / collision_waypoints (simplecars.jl:55-82) behind is_free_motion
 *   (statespaces.jl:134-142, 153-158).
 * sin / cos / atan2 / acos are fixed polynomial routines (specified in oracle/cars.c; the reference calls openlibm:
 * parity unpinned there); everything else follows the reference's operation order. */
#define MPB200_CAR_REEDS_SHEPP 0
#define MPB200_CAR_DUBINS 1
/* tableF column v: { i != v : (x,y) within r, chopped d(V[v] -> V[i]) <= r }, stored value = the path length;
 * tableB column v: the same with d(V[i] -> V[v]) (Dubins; pass tableB = NULL for the symmetric Reeds-Shepp
 * metric, whose MetricNN serves inballF! and inballB! from the forward table).  chopval = the metric's chop value
 * (setup_steering sets it to r).  s must hold d = 3 states; the query range of s is honoured. */
int mpb200_car_inball_build(mpb200_samples *s, int32_t kind, double turning_radius, double r, double chopval,
                            mpb200_table **tableF, mpb200_table **tableB, int64_t *nnzF, int64_t *nnzB);
/* entries of the (x, y) candidate table behind the last mpb200_car_inball_build on s = pairs whose exact metric was
 * evaluated (per direction); measurement aid */
int mpb200_car_last_candidates(const mpb200_samples *s, int64_t *pairs);
/* (cost, steering_control) for n explicit pairs: segments = n x 5 x (duration, signed speed, signed curvature),
 * nseg[i] of them valid (3 for Dubins, 3..5 for Reeds-Shepp) */
int mpb200_car_steer(int32_t kind, double turning_radius, double speed, const double *v_aos, const double *w_aos,
                     int64_t n, double *cost, int32_t *nseg, double *segments);
/* is_free_motion(V[y], V[x], CC, SS) for every stored entry (row y, column x) of a table: arc waypoints every pi/12
 * of positive heading change (simplecars.jl:71-82), each but the last bounds-checked, consecutive ones swept. */
int mpb200_car_edges_free(const mpb200_samples *s, const mpb200_table *t, int32_t kind, double turning_radius,
                          double speed, const mpb200_obstacles *o, const mpb200_space_desc *ss, uint64_t *bitchunks,
                          int64_t *checks);
int mpb200_car_motions_free(int32_t kind, double turning_radius, double speed, const double *v_aos,
                            const double *w_aos, int64_t n, const mpb200_obstacles *o, const mpb200_space_desc *ss,
                            uint8_t *out, int64_t *checks);

/* ---- Monte-Carlo trajectory collision probability -----------------------------------
 * NOT in the reference (only paper links, README.md:9-10, and the helper geometry
 * closest/closeR, SAT2D.jl:208-285, boxesND.jl:61-86): specified in SURVEY.md section 11 /
 * DESIGN.md.  Closed loop z' = F_t z + G_t eps_t (z_0 = 0), workspace w_t = wbar_t + Wz z_t,
 * hit = some w_t (swept: some segment w_{t-1}->w_t) collides with the obstacle set, defensive
 * mixture proposal over the stacked noise, Philox4x32-10 keyed by (seed, rollout id).
 * All matrices row-major. */
typedef struct {
    int32_t T;           /* steps */
    int32_t nz;          /* closed-loop state dimension */
    int32_t q;           /* noise dimension per step */
    int32_t dw;          /* workspace dimension */
    const double *F;     /* T x nz x nz */
    const double *G;     /* T x nz x q */
    const double *Wz;    /* dw x nz */
    const double *wbar;  /* (T+1) x dw nominal workspace points (index 0 = start, never tested as a point) */
    int32_t K;           /* shifted mixture components (besides the nominal one) */
    const double *alpha; /* K+1 mixture weights, alpha[0] = nominal, sum 1 */
    const double *mu;    /* K x (T*q) mean shifts of the stacked noise */
    int32_t swept;       /* 0: point test per step, 1: segment test between consecutive steps */
} mpb200_mc_problem;
typedef struct {
    double s1;    /* sum of w * hit          */
    double s2;    /* sum of (w * hit)^2      */
    double s0;    /* sum of w (diagnostic: -> n) */
    int64_t n;    /* rollouts                */
    int64_t hits; /* unweighted hit count    */
} mpb200_mc_result;
/* Rollout ids [first, first + n): the shard of one GPU; sums of shards add up to the whole.
 * hit_out (n bytes) / w_out (n doubles) are optional per-rollout outputs. */
int mpb200_mc_collision_probability(const mpb200_mc_problem *p, const mpb200_obstacles *o, uint64_t seed,
                                    int64_t first, int64_t n, mpb200_mc_result *out, uint8_t *hit_out,
                                    double *w_out);

/* ---- k-nearest connections ---------------------------------------------------------------------
 * The reference exports knn / knnF / knnB / mutualknn* (nearneighbors.jl:9-11) and FMT*'s connections = :K branch
 * calls mutualknnF! / knnB! (fmt.jl:6,17-19,70,72), but defines none of them (`:K` throws there).  Specification
 * implemented here (parity unpinned; restated in oracle/oracle.py):
 *   knn(v, k): the k samples j != v with the smallest stored value, ties towards the smaller index, returned like
 *   every neighbourhood (ascending indices + values);  mutualknnF(v, k) = knnF(v, k) U { w : v in knnB(w, k) }.
 * Both are table operations on top of ANY neighbour table (Euclidean or steering cost):
 *   mpb200_table_knn keeps the k best entries of every column of t; columns of t with fewer than k entries are kept
 *   whole and counted in *short_cols -- rebuild t with a larger radius until it is 0 and the result is the k-NN table;
 *   mpb200_table_union_transpose forms out[:, v] = a[:, v] U { w : v in b[:, w] } (values from a, else from b;
 *   full-range tables over the same sample set).  Columns are limited to 8192 entries.
 * Non-NULL *out handles are reused.  Edge validity works on the results like on any table. */
int mpb200_table_knn(const mpb200_table *t, int k, mpb200_table **out, int64_t *nnz, int64_t *short_cols);
/* only the question "does every column of t hold at least k entries?": *short_cols = columns that do not */
int mpb200_table_short_columns(const mpb200_table *t, int k, int64_t *short_cols);
int mpb200_table_union_transpose(const mpb200_table *a, const mpb200_table *b, mpb200_table **out, int64_t *nnz);

/* ---- closest obstacle points under a weight matrix (Monte-Carlo proposal geometry) ----------
 * Replaces closest(p, shape, W) / closeR(p, CC, W, r2) (SAT2D.jl:208-285; boxesND.jl:61-86; robots2D.jl:25-26)
 * for n query points at once, each with its own SPD weight matrix W_i (dw x dw row-major; dw = 2 for 2-D
 * obstacle sets, = box dimension <= 4 for box lists).  S = number of basic shapes (circles + polygons, or boxes).
 * Per point: count[i] shapes lie closer than r2 (squared W-distance); d2 / shape / x list them in ascending
 * d2 (ties in shape order), capacity S per point: d2[i*S + k], shape[i*S + k], x[(i*S + k)*dw ..].
 * all_d2 / all_x (optional, n x S [x dw]) receive closest() for every basic shape, unsorted. */
int mpb200_close_points(const mpb200_obstacles *o, const double *p_aos, const double *W, int64_t n, int dw, double r2,
                        int32_t *count, double *d2, int32_t *shape, double *x, double *all_d2, double *all_x);

/* ---- multi-GPU exchange by direct peer stores (one process per GPU, one box) ----------
 * The reference has no distributed layer; this is the exchange step of the query-range-sharded
 * precompute (DESIGN.md section 8): after a rank has built its table shard and the validity of its
 * edges, ONE call stores the shard's int32 column lengths and validity words into slot `rank` of
 * every peer's receive buffer over NVLink (CUDA IPC mapped memory, no NCCL, no staging copies) and
 * runs a device-side flag barrier, all stream-ordered and asynchronous.
 *   create  -> allocates this rank's receive buffer (2 alternating sets x world slots) and returns
 *              its 64-byte CUDA IPC handle; the caller exchanges the handles of all ranks by any
 *              means (torch.distributed all_gather, MPI, a file) and hands them to connect.
 *   push    -> enqueue pack + peer stores + barrier for the current contents of `t`
 *              (needs mpb200_edges_free / mpb200_lq_edges_free on it first).
 *   view    -> device pointer of the newest complete set: world slots of slot_bytes each;
 *              slot g = [int64 ncols, int64 nnz, int64 epoch, pad to 64 B | int32 counts at
 *              counts_off | uint64 validity words at words_off].  With status != NULL the call
 *              waits for the enqueued pushes and returns 0, or 1 + the rank that never arrived.
 * A set stays valid until this rank's second-next push. */
typedef struct mpb200_xchg mpb200_xchg;
#define MPB200_IPC_HANDLE_BYTES 64
#define MPB200_XCHG_MAX_WORLD 16
int mpb200_xchg_create(int rank, int world, int64_t max_ncols, int64_t word_cap, mpb200_xchg **out, void *ipc_handle);
int mpb200_xchg_connect(mpb200_xchg *x, const void *handles /* world x 64 bytes, rank order */);
/* Optional: tie a table handle to the exchange.  Every later mpb200_inball_build on it starts sending the column
 * lengths of the coming epoch right after its count scan, on a side stream underneath the fill and validity
 * kernels; the following mpb200_xchg_push then only sends the validity words.  x = NULL detaches. */
int mpb200_xchg_attach(mpb200_xchg *x, mpb200_table *t);
int mpb200_xchg_push(mpb200_xchg *x, const mpb200_table *t);
int mpb200_xchg_view(const mpb200_xchg *x, void **recv, int64_t *slot_bytes, int64_t *counts_off, int64_t *words_off,
                     int64_t *status);
int mpb200_xchg_destroy(mpb200_xchg *x);

/* ---- measured arithmetic-pipe peaks (roofline denominators for the FP64 / FP32 kernels) ----
 * Runs a register-resident instruction stream on every SM and returns operations per second
 * (an FMA counts as two), CUDA-event timed.  DADD_DMUL is the no-FMA rate the parity kernels
 * are bound by (one rounding per operation, as the reference computes). */
#define MPB200_PEAK_DADD_DMUL 0
#define MPB200_PEAK_DFMA 1
#define MPB200_PEAK_FFMA 2
int mpb200_pipe_peak(int kind, double *ops_per_s);
/* Duration (ms, CUDA events, best of 3 after an L2 eviction) of a kernel that does nothing but WRITE a table of
 * t's shape: every column as one contiguous Int64 + one Float64 burst at colptr[w], columns visited in the order the
 * fill kernel visits them, constant data.  This is what the reference's CSC output format costs on the device before
 * any neighbour work: the floor the fill kernel's time is compared with, next to the plain-copy HBM peak. */
int mpb200_table_write_floor(const mpb200_table *t, double *ms);

/* ---- planning on the device: group-marching FMT* (GMT*; Ichter, Schmerling & Pavone 2017) -------------------
 * Plans over tables and validity bits that are already on the device, so nothing N-sized crosses PCIe on the way in.
 * Inputs: samples 1..N of s; fwd (DF: column z holds the x with an edge z -> x); bwd (DB: column x holds the y with
 * an edge y -> x and its cost) with its edge bits (the last mpb200_edges_free / _lq_ / _car_ result on bwd); the
 * point bits of s (the last mpb200_points_free) when checkpts != 0, else every sample counts as free; a goal mask;
 * a width w = lambda * r.
 * State: C (cost), A (parent, 0 = none), status W (unvisited) / H (open) / closed.  Initially only init is in H, C = 0.
 * Each iteration:
 *   1. H empty: failed.  Else thr = min_{y in H} C[y] + w (one FP64 add), group G = { y in H : C[y] <= thr }.
 *   2. G holds a goal vertex: solved; the result is the goal vertex of G with the smallest (C, index).
 *   3. candidates X = { x in column g of DF for some g in G : x in W, free(x) }.
 *   4. every x in X, against the state at the start of the iteration: among the entries e of column x of DB whose
 *      row y is in H (G included), none -> skip x; else e* = the first in storage order minimising C[y] + nzval[e]
 *      (one FP64 add); count one check (and one in checks_in_bounds when V[y] lies in the space bounds); if the
 *      edge bit of e* is set: A[x] = y, C[x] = that cost, x joins H_new.
 *   5. G becomes closed, H_new joins H.
 * At w = 0 with no two open vertices of equal cost, G is the vertex FMT*'s heap would dequeue: tree, cost, path and
 * check count equal fmtstar's.  Every output is a function of sets: identical for every run and launch geometry.
 * One cooperative kernel runs the whole loop (no host round trip per iteration); MPB200_GMT_GRID=<blocks> forces its
 * grid size (clamped to the co-resident maximum).
 * Rejected with MPB200_EARG: tables built from another sample set or over a query range other than [0, N), missing
 * or stale edge bits on bwd, checkpts without full-range point bits of s. */
typedef struct {
    const mpb200_table *fwd;        /* DF */
    const mpb200_table *bwd;        /* DB, with current edge bits */
    const uint64_t *goal_bits;      /* host BitVector chunks, ceil(N/64) words: goal mask */
    int64_t init;                   /* 1-based */
    double width;                   /* w = lambda * r, >= 0 */
    int32_t checkpts;               /* 0: every sample counts as free */
    const mpb200_space_desc *space; /* optional (NULL: checks_in_bounds = 0): bounds for checks_in_bounds */
} mpb200_gmt_desc;
typedef struct {
    int32_t solved;
    int32_t grid_blocks;        /* blocks of the cooperative launch */
    int64_t goal;               /* 1-based goal vertex reached, 0 when failed */
    double cost;                /* C[goal], +inf when failed */
    int64_t iterations;         /* groups expanded */
    int64_t expansions;         /* sum of |G| over them */
    int64_t checks;             /* edge-bit lookups (step 4) */
    int64_t checks_in_bounds;   /* of those, with V[y] inside the space bounds */
    int64_t path_len;           /* vertices init .. goal, 0 when failed */
} mpb200_gmt_result;
/* path: path_len 1-based vertices init .. goal, written only when path_len <= path_cap (path may be NULL when
 * path_cap == 0); tree (N int64, parents, 1-based, 0 = none) and costs (N f64) may be NULL.  Waits for the result. */
int mpb200_gmt_plan(const mpb200_samples *s, const mpb200_gmt_desc *desc, mpb200_gmt_result *res, int64_t *path,
                    int64_t path_cap, int64_t *tree, double *costs);

/* Lazy GMT*: the same plan without edge bits.  Step 4 reads
 *      if is_free_motion(V[y], V[x], CC, SS): A[x] = y, C[x] = that cost, x joins H_new
 * with the motion check evaluated inside the planning kernel, on e* only; everything else (the decision point, the
 * argmin, the counters) is as above, so for the same tables the result equals mpb200_gmt_plan's over bits computed for
 * the same obstacles, byte for byte.  The motion check is the one the matching edge pass runs: a straight segment
 * (as mpb200_edges_free), the optimal LQ trajectory (as mpb200_lq_edges_free, steering horizon r) or the car path
 * (as mpb200_car_edges_free).  *segment_checks (may be NULL) = segment tests those checks ran, each preceded by the
 * bounds test of its first waypoint and stopping at the first failure, the last waypoint never bounds-checked: the
 * increment of the reference's CC.count.  For straight segments it equals checks_in_bounds.
 * desc->space is required (the space of the motion check and of checks_in_bounds).  The edge bits of bwd are never
 * read, required or changed.  Rejected with MPB200_EARG: everything mpb200_gmt_plan rejects but the edge-bit check;
 * NULL edges or obstacles, an unknown kind; no space; a car kind with d != 3, an unknown car kind, turning radius or
 * speed not positive and finite; an LQ kind without a system, with a d that does not match it, or r not positive and
 * finite; an obstacle / workspace combination the matching *_edges_free rejects.  One launch per plan. */
#define MPB200_GMT_EDGES_STRAIGHT 0   /* as mpb200_edges_free     */
#define MPB200_GMT_EDGES_LQ       1   /* as mpb200_lq_edges_free  */
#define MPB200_GMT_EDGES_CAR      2   /* as mpb200_car_edges_free */
typedef struct {
    int32_t kind;                       /* MPB200_GMT_EDGES_* */
    const mpb200_obstacles *obstacles;
    const mpb200_lq *lq;                /* kind LQ */
    double r;                           /* kind LQ: steering horizon, the r mpb200_lq_edges_free takes */
    int32_t car_kind;                   /* kind CAR: MPB200_CAR_REEDS_SHEPP / MPB200_CAR_DUBINS */
    double turning_radius, speed;       /* kind CAR */
} mpb200_gmt_edges;
int mpb200_gmt_plan_lazy(const mpb200_samples *s, const mpb200_gmt_desc *desc, const mpb200_gmt_edges *edges,
                         mpb200_gmt_result *res, int64_t *segment_checks, int64_t *path, int64_t path_cap,
                         int64_t *tree, double *costs);

/* A batch of GMT* queries over one roadmap: nq independent plans over the same samples, the same fwd / bwd tables,
 * point bits, checkpts setting and space, and the same edge test (edges == NULL: the edge bits of bwd, as
 * mpb200_gmt_plan; else the motion check of edges, as mpb200_gmt_plan_lazy).  Query q has its own init, goal mask
 * and width from descs[q].  Every output of query q (res[q] but grid_blocks, segment_checks[q], row q of paths,
 * trees and costs) is byte-identical to what mpb200_gmt_plan / _lazy returns for descs[q] alone over the same tables,
 * whatever the other queries of the batch, their order or the grid size.  grid_blocks is that of the one launch.
 * The queries march in lockstep through one cooperative launch and share its grid-wide barriers; measured at C2 on one
 * B200 (DESIGN.md section 10b), 16 queries cost 2.8x less than their single plans and 64 queries 4x less, and a batch
 * lasts as long as its longest query.
 * paths: nq x path_cap, row q = the path of query q, written only when its path_len <= path_cap (paths may be NULL
 * when path_cap == 0); trees (int64) and costs (f64): nq x N each, row q = query q, may be NULL.
 * Rejected with MPB200_EARG before any launch: everything mpb200_gmt_plan / _lazy rejects, for every query; nq < 1;
 * NULL descs or res; descs whose fwd, bwd, checkpts or space differ from those of descs[0]; NULL paths with
 * path_cap > 0.  MPB200_ENOMEM, without a launch, when the scratch of the batch cannot be reserved: per query
 * MPB200_GMT_BATCH_BYTES_PER_QUERY(N, path_cap) bytes of device memory (C, A, status, four (query, vertex) lists, the
 * path row, the goal mask, the control block).  One launch per call, timed under MPB200_OP_PLAN. */
#define MPB200_GMT_BATCH_BYTES_PER_QUERY(N, path_cap) \
    (52 * (int64_t)(N) + 8 * ((int64_t)(path_cap) < (int64_t)(N) ? (int64_t)(path_cap) : (int64_t)(N)) + \
     8 * (((int64_t)(N) + 63) / 64) + 120)
int mpb200_gmt_plan_batch(const mpb200_samples *s, const mpb200_gmt_desc *descs, int64_t nq,
                          const mpb200_gmt_edges *edges, mpb200_gmt_result *res, int64_t *segment_checks,
                          int64_t *paths, int64_t path_cap, int64_t *trees, double *costs);

/* ---- shortcutting planned paths: the cheapest collision-free route through a path's subdivided waypoints ----------
 * Not the reference's shortcut / adaptive_shortcut! (postprocessors.jl, not in the tree): specified here, restated in
 * tests/oracle_shortcut.py.  npaths >= 1 paths, each handled on its own: path q is the states Y[0..L-1] (AoS, d doubles
 * each) at rows offsets[q] .. offsets[q+1]-1 of states_aos (offsets[0] = 0, L = offsets[q+1] - offsets[q] >= 1).
 *   1. Nodes: M = (L-1) k + 1 with k = subdivisions.  Node i k is Y[i] bit for bit; for m = 1..k-1 node i k + m is
 *      Y[i]_c + t (Y[i+1]_c - Y[i]_c) with t = (double)m / (double)k, every operation rounded on its own (no FMA).
 *   2. Visibility: for every pair a < b, free(a, b) = is_free_motion(node a, node b) with straight waypoints, the
 *      predicate of mpb200_segments_free / mpb200_edges_free: node a is bounds-checked, node b is not.
 *      segment_checks[q] = pairs whose segment test ran (node a in bounds; the CC.count increment);
 *      pairs[q] = M (M-1) / 2.
 *   3. Cost: cost(a, b) = sqrt(sum_c (node a_c - node b_c)^2), summed in index order, no FMA (the r-ball table's value).
 *   4. Minimum: best[0] = +0.0; for b = 1..M-1, best[b] = min over free(a, b) of best[a] + cost(a, b) (one FP64 add),
 *      pred[b] = the smallest a attaining it (the longest jump: collinear subdivision nodes drop out when costs tie);
 *      +inf when no a gives a finite value.
 *   5. Output: best[M-1] finite: the nodes of the pred chain 0 .. M-1, costs[q] = best[M-1].  Otherwise (the path was
 *      not free): the input path unchanged, costs[q] = +inf.  L = 1: the input state, cost 0, 0 pairs.
 * Guarantees:
 *   - If every consecutive motion of the input is free -- true of every fmtstar / gmtstar / gmtstar_batch solution under
 *     the same obstacles and space, whose planner tested exactly those endpoints in that direction -- the output cost
 *     is <= the input's edge costs summed in path order, which is the planner's C[goal] bit for bit (the input edges
 *     are edges of the minimum's DAG with the same cost formula, and FP64 addition is monotone).
 *   - Every consecutive motion of the output is free: calling again on the output is valid and never raises the cost.
 *   - The outputs of path q are byte-identical whatever else is in the call, in whatever order, on whatever grid
 *     (MPB200_SHORTCUT_GRID=<blocks> forces the visibility pass's grid, clamped to the co-resident maximum).
 * Outputs: out_len[q] and costs[q] always; row q of out_states (npaths x out_cap x d) only when out_len[q] <= out_cap;
 * pairs and segment_checks may be NULL.  Waits for its results.
 * Rejected with MPB200_EARG before any launch: npaths < 1; NULL states, offsets, out_len or costs; offsets not strictly
 * increasing from 0 (a path with L = 0); subdivisions < 1; a path with M > MPB200_SHORTCUT_MAX_NODES; NULL out_states
 * with out_cap > 0; out_cap < 0; a (d, workspace) / obstacle combination mpb200_segments_free rejects.  MPB200_ENOMEM,
 * without a launch, when the scratch cannot be reserved (per path M ceil(M / 32) 4 bytes of visibility bits, about M^2 / 8, plus 16 d + 12 bytes per node).
 * Three launches per call whatever npaths, timed under MPB200_OP_PATH (phase 1: nodes and visibility; phase 2: the
 * minimum and the output rows). */
#define MPB200_SHORTCUT_MAX_NODES 32768
int mpb200_shortcut_paths(const double *states_aos, const int64_t *offsets, int64_t npaths, int d,
                          const mpb200_obstacles *o, const mpb200_space_desc *ss, int32_t subdivisions,
                          double *out_states, int64_t out_cap, int64_t *out_len, double *costs,
                          int64_t *pairs, int64_t *segment_checks);

#ifdef __cplusplus
}
#endif
#endif
