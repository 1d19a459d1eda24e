// api.cu -- the extern "C" entry points declared in include/mpb200.h, plus the runtime
// plumbing (context, error strings, growing device buffers, event timing).
#include "common.cuh"
#include "predicates.cuh"
#include <climits>
#include <cstdio>
#include <cstring>
#include <limits>
#include <algorithm>
#include <emmintrin.h>
#include <new>
#include <thread>
#include <vector>

namespace mpb {

Context &ctx() {
    static Context c;
    return c;
}

static thread_local char g_err[512] = "";
void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

// ---- device memory: DevBuf over a block cache ------------------------------------------------
// cudaMalloc / cudaFree of the few-hundred-MB arrays of a table cost milliseconds each (and cudaFree
// synchronises the device), which dwarfs the sub-millisecond kernels when a caller creates and drops
// sample sets and tables per planning step.  Released blocks are therefore parked in a free list and
// handed back by best fit.  Everything the library enqueues goes to ONE stream at a time
// (mpb200_set_stream synchronises the old one), so a parked block can be reused without waiting: its
// next user is ordered after its last one.
namespace {
struct Block { void *p; size_t cap; };
std::vector<Block> g_blocks;
size_t g_cached_bytes = 0;
constexpr size_t kCacheLimit = size_t(64) << 30;  // beyond this, released blocks go back to the driver

void *cache_take(size_t bytes, size_t *cap) {
    int best = -1;
    for (int i = 0; i < (int)g_blocks.size(); ++i) {
        const size_t c = g_blocks[i].cap;
        if (c >= bytes && c <= 2 * bytes + (size_t(1) << 20) && (best < 0 || c < g_blocks[best].cap)) best = i;
    }
    if (best < 0) return nullptr;
    void *p = g_blocks[best].p;
    *cap = g_blocks[best].cap;
    g_cached_bytes -= *cap;
    g_blocks[best] = g_blocks.back();
    g_blocks.pop_back();
    return p;
}
}  // namespace

size_t cache_parked_bytes() { return g_cached_bytes; }

uint64_t next_serial() {
    static uint64_t n = 0;
    return ++n;
}

void cache_release_all() {
    for (const Block &b : g_blocks) cudaFree(b.p);
    g_blocks.clear();
    g_cached_bytes = 0;
}

int DevBuf::reserve(size_t bytes) {
    if (bytes <= cap) return 0;
    release();
    // grow geometrically so repeated builds with slightly different sizes settle quickly
    size_t want = bytes + bytes / 8 + 256;
    if ((p = cache_take(bytes, &cap))) return 0;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {  // give the parked blocks back to the driver and ask for the exact size
        cudaGetLastError();
        cudaStreamSynchronize(ctx().stream);
        cache_release_all();
        e = cudaMalloc(&p, bytes);
        want = bytes;
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        p = nullptr;
        cap = 0;
        return fail(MPB200_ENOMEM, "cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
    }
    cap = want;
    return 0;
}
void DevBuf::release() {
    if (p) {
        if (ctx().ready && g_cached_bytes + cap <= kCacheLimit) {
            g_blocks.push_back({p, cap});
            g_cached_bytes += cap;
        } else {
            cudaFree(p);
        }
    }
    p = nullptr;
    cap = 0;
}

namespace {
struct TraceRec { cudaEvent_t ev; const char *file; int line; };
std::vector<TraceRec> g_trace;
size_t g_trace_n = 0;
const bool g_trace_on = getenv("MPB200_TRACE") != nullptr;
}  // namespace
void trace_mark(const char *file, int line) {
    if (!g_trace_on) return;
    if (g_trace_n == g_trace.size()) {
        TraceRec r{nullptr, file, line};
        cudaEventCreate(&r.ev);
        g_trace.push_back(r);
    }
    g_trace[g_trace_n].file = file;
    g_trace[g_trace_n].line = line;
    cudaEventRecord(g_trace[g_trace_n].ev, ctx().stream);
    ++g_trace_n;
}
void trace_dump() {
    if (!g_trace_on || g_trace_n == 0) return;
    cudaStreamSynchronize(ctx().stream);
    for (size_t i = 0; i < g_trace_n; ++i) {
        float ms = 0;
        if (i) cudaEventElapsedTime(&ms, g_trace[i - 1].ev, g_trace[i].ev);
        const char *f = strrchr(g_trace[i].file, '/');
        fprintf(stderr, "[trace] %-18s:%-4d +%8.1f us\n", f ? f + 1 : g_trace[i].file, g_trace[i].line, ms * 1e3);
    }
    g_trace_n = 0;
}

int phase_mark(int i) {
    Context &c = ctx();
    if (i < 0 || i > kMaxPhases) return 0;
    trace_mark("phase", i);
    cudaEventRecord(c.ev[c.bank][i], c.stream);
    return 0;
}
void phase_bank(int op) {
    if (op >= 0 && op < kBanks) ctx().bank = op;
}
int phases_collect(int n) {
    Context &c = ctx();
    c.pending_marks[c.bank] = n;  // resolved lazily by phases_resolve(): the API call itself does not wait for the GPU
    return 0;
}
static void phases_resolve(int b) {
    Context &c = ctx();
    const int n = c.pending_marks[b];
    if (n <= 0) return;
    c.pending_marks[b] = 0;
    cudaEventSynchronize(c.ev[b][n]);
    for (int k = 0; k < kMaxPhases; ++k) c.last_ms[b][k] = 0;
    float ms = 0;
    if (cudaEventElapsedTime(&ms, c.ev[b][0], c.ev[b][n]) == cudaSuccess) c.last_ms[b][0] = ms;
    for (int k = 0; k < n && k + 1 < kMaxPhases; ++k)
        if (cudaEventElapsedTime(&ms, c.ev[b][k], c.ev[b][k + 1]) == cudaSuccess) c.last_ms[b][k + 1] = ms;
    cudaGetLastError();
}

// implemented in the kernel translation units
int compute_bbox(mpb200_samples *s, int64_t j0, int64_t j1);
int check_sorted_x(mpb200_samples *s, int *d_flag);
int sample_free_device(const mpb200_obstacles *o, const mpb200_space_desc *ss, int64_t n_want, uint64_t seed,
                       double *dV, DevBuf &scratch, DevBuf &tmp, int64_t *h_used);
int morton_reorder_device(double *dV, int64_t N, const mpb200_space_desc *ss, DevBuf &scratch);
int grid_inball_build(mpb200_samples *s, double r, mpb200_table *t);
int brute_inball_build(mpb200_samples *s, double r, mpb200_table *t);

int points_free_device(const double *dV, int64_t n, int d, const mpb200_obstacles *o, const mpb200_space_desc *ss,
                       uint32_t *d_bits32, uint8_t *d_bytes, const mpb200_samples *cell_order = nullptr);
int edges_free_device(const mpb200_samples *s, mpb200_table *t, const mpb200_obstacles *o,
                      const mpb200_space_desc *ss, uint32_t *d_bits32, unsigned long long *d_counters);
int segments_free_device(const double *dA, const double *dB, int64_t n, int d, const mpb200_obstacles *o,
                         const mpb200_space_desc *ss, uint8_t *d_out);

int lq_inball_build(mpb200_samples *s, const mpb200_lq *lq, double r, mpb200_table *tF, mpb200_table *tB);
int lq_steer_device(const mpb200_lq *lq, const double *dA, const double *dB, int64_t n, double r, double *d_cost,
                    double *d_topt);
int lq_edges_free_device(const mpb200_samples *s, const mpb200_table *t, const mpb200_lq *lq, double r,
                         const mpb200_obstacles *o, const mpb200_space_desc *ss, uint32_t *d_bits32,
                         unsigned long long *d_checks);
int lq_motions_free_device(const mpb200_lq *lq, double r, const double *dA, const double *dB, int64_t n, int d_state,
                           const mpb200_obstacles *o, const mpb200_space_desc *ss, uint8_t *d_out,
                           unsigned long long *d_checks);

int car_args(int32_t kind, double rturn, double speed);
int car_extract_xy_device(const double *dV3, int64_t N, double *dV2);
int car_inball_device(const mpb200_samples *s, const mpb200_table *cand, int kind, double rturn, double r, double chopval,
                      mpb200_table *tF, mpb200_table *tB, DevBuf &work, DevBuf &scan_tmp);
int car_edges_free_device(const mpb200_samples *s, const mpb200_table *t, int kind, double rturn, double speed,
                          const mpb200_obstacles *o, const mpb200_space_desc *ss, uint32_t *d_bits32,
                          unsigned long long *d_checks);
int car_motions_free_device(int kind, double rturn, double speed, const double *dA, const double *dB, int64_t n,
                            const mpb200_obstacles *o, const mpb200_space_desc *ss, uint8_t *d_out, unsigned long long *d_checks);
int car_steer_device(int kind, double rturn, double speed, const double *dA, const double *dB, int64_t n, double *d_cost,
                     int *d_nseg, double *d_segs);
int pipe_peak_device(int kind, double *ops_per_s);
int table_knn_device(const mpb200_table *t, int k, mpb200_table *out, int64_t *short_cols, DevBuf &scan_tmp);
int table_short_columns_device(const mpb200_table *t, int k, int64_t *short_cols);
int table_union_transpose_device(const mpb200_table *a, const mpb200_table *b, mpb200_table *out, DevBuf &scan_tmp);
int table_write_floor_device(const mpb200_table *t, double *ms);
int close_points_device(const mpb200_obstacles *o, const double *dP, const double *dW, int64_t n, int dw, double r2,
                        int *d_count, double *d_d2, int *d_shape, double *d_x, double *d_all_d2, double *d_all_x);
int lqg_setup_host(int n, int m, const double *A, const double *B, const double *c, const double *R, LqgHost *S);
int lqg_upload(mpb200_lq *lq);
int lqg_inball_build(mpb200_samples *s, const mpb200_lq *lq, double r, mpb200_table *tF, mpb200_table *tB);
int lqg_steer_device(const mpb200_lq *lq, const double *dA, const double *dB, int64_t n, double r, double *d_cost,
                     double *d_topt);
int lqg_edges_free_device(const mpb200_samples *s, const mpb200_table *t, const mpb200_lq *lq, double r,
                          const mpb200_obstacles *o, const mpb200_space_desc *ss, uint32_t *d_bits32,
                          unsigned long long *d_checks);
int lqg_motions_free_device(const mpb200_lq *lq, double r, const double *dA, const double *dB, int64_t n, int d_state,
                            const mpb200_obstacles *o, const mpb200_space_desc *ss, uint8_t *d_out,
                            unsigned long long *d_checks);
int mc_run_device(const mpb200_mc_problem *p, const mpb200_obstacles *o, unsigned long long seed, long long first,
                  long long n, double *h_out4, uint8_t *h_hit, double *h_w);

}  // namespace mpb

using namespace mpb;

static void release_fetch_staging();

extern "C" {

int mpb200_version(void) { return 100; }

const char *mpb200_last_error(void) { return g_err; }

int mpb200_init(int device) {
    Context &c = ctx();
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(MPB200_ECUDA, "no CUDA device available (%s); libmpb200 has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= ndev) return fail(MPB200_EARG, "device %d out of range (0..%d)", device, ndev - 1);
    if (c.ready && c.device == device) return MPB200_OK;
    if (c.ready) mpb200_shutdown();
    MPB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    MPB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(MPB200_ECUDA, "device %d (%s) is compute capability %d.%d; libmpb200 is built for sm_100a only",
                    device, prop.name, prop.major, prop.minor);
    c.device = device;
    c.sm_count = prop.multiProcessorCount;
    MPB_CUDA(cudaStreamCreateWithFlags(&c.own_stream, cudaStreamNonBlocking));
    c.stream = c.own_stream;
    for (int b = 0; b < kBanks; ++b)
        for (int i = 0; i <= kMaxPhases; ++i) MPB_CUDA(cudaEventCreate(&c.ev[b][i]));
    MPB_CUDA(cudaEventCreateWithFlags(&c.ev_scalar, cudaEventDisableTiming));
    MPB_CUDA(cudaMalloc(&c.d_scalar, sizeof(int64_t) * 16));
    MPB_CUDA(cudaMemset(c.d_scalar, 0, sizeof(int64_t) * 16));  // slots are read back in groups; none is ever undefined
    MPB_CUDA(cudaMallocHost(&c.h_scalar, sizeof(int64_t) * 16));
    c.launches = 0;
    c.ready = true;
    return MPB200_OK;
}

void mpb200_shutdown(void) {
    Context &c = ctx();
    if (!c.ready) return;
    cudaDeviceSynchronize();
    for (int b = 0; b < kBanks; ++b)
        for (int i = 0; i <= kMaxPhases; ++i)
            if (c.ev[b][i]) cudaEventDestroy(c.ev[b][i]), c.ev[b][i] = nullptr;
    cache_release_all();
    release_fetch_staging();
    if (c.ev_scalar) cudaEventDestroy(c.ev_scalar), c.ev_scalar = nullptr;
    if (c.d_scalar) cudaFree(c.d_scalar), c.d_scalar = nullptr;
    if (c.h_scalar) cudaFreeHost(c.h_scalar), c.h_scalar = nullptr;
    if (c.own_stream) cudaStreamDestroy(c.own_stream), c.own_stream = nullptr;
    c.stream = nullptr;
    c.ready = false;
}

int mpb200_set_stream(void *cuda_stream) {
    MPB_REQUIRE_INIT();
    Context &c = ctx();
    MPB_CUDA(cudaStreamSynchronize(c.stream));
    c.stream = cuda_stream ? reinterpret_cast<cudaStream_t>(cuda_stream) : c.own_stream;
    return MPB200_OK;
}
int mpb200_synchronize(void) {
    MPB_REQUIRE_INIT();
    MPB_CUDA(cudaStreamSynchronize(ctx().stream));
    trace_dump();
    return MPB200_OK;
}
int mpb200_release_cached(void) {
    MPB_REQUIRE_INIT();
    MPB_CUDA(cudaStreamSynchronize(ctx().stream));
    cache_release_all();
    return MPB200_OK;
}
int mpb200_host_alloc(uint64_t bytes, void **out) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(out != nullptr, "out is NULL");
    *out = nullptr;
    MPB_CUDA(cudaMallocHost(out, bytes ? bytes : 1));
    return MPB200_OK;
}
int mpb200_host_free(void *p) {
    if (p) MPB_CUDA(cudaFreeHost(p));
    return MPB200_OK;
}
int64_t mpb200_launch_count(void) { return ctx().launches; }
double mpb200_last_ms_of(int op, int phase) {
    if (op < 0 || op >= kBanks || phase < 0 || phase >= kMaxPhases) return 0;
    if (ctx().ready) phases_resolve(op);
    return ctx().last_ms[op][phase];
}
double mpb200_last_ms(int phase) { return mpb200_last_ms_of(ctx().bank, phase); }

// Host -> device copy ordered on the library's stream (the block cache hands out parked blocks without
// waiting, on the premise that ALL buffer traffic is on that one stream), complete on return: the source
// may be a temporary.
static int upload_sync(void *dst, const void *src, size_t bytes) {
    cudaStream_t st = ctx().stream;
    MPB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    return MPB200_OK;
}

// ---- samples -----------------------------------------------------------------------
// bounding box + x-sortedness of a sample set whose V is already on the device; leaves the stream idle
static int finish_samples(mpb200_samples *s) {
    Context &c = ctx();
    cudaStream_t st = c.stream;
    const int d = s->d;
    if (s->N > 0) {
        if (int rc = compute_bbox(s, 0, s->N)) return rc;
        MPB_CUDA(cudaMemcpyAsync(s->h_bbox, s->minmax.p, sizeof(double) * 2 * d, cudaMemcpyDeviceToHost, st));
        // samples ordered along x (e.g. stored in stripe order for sharding)?  Then a shard's grid build only
        // has to look at its own stripe of the array.
        if (int rc = check_sorted_x(s, reinterpret_cast<int *>(c.d_scalar + 8))) return rc;
        MPB_CUDA(cudaMemcpyAsync(c.h_scalar + 8, c.d_scalar + 8, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    }
    MPB_CUDA(cudaStreamSynchronize(st));
    if (s->N > 0) s->sorted_x = *reinterpret_cast<int *>(c.h_scalar + 8) == 0;
    memcpy(s->h_qbbox, s->h_bbox, sizeof(s->h_bbox));
    return MPB200_OK;
}
int mpb200_samples_create(const double *V_aos, int64_t N, int d, mpb200_samples **out) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(out != nullptr, "out is NULL");
    MPB_CHECK_ARG(N >= 0 && N < INT_MAX, "N out of range");
    MPB_CHECK_ARG(d >= 1 && d <= kMaxDim, "d out of range (1..16)");
    MPB_CHECK_ARG(V_aos != nullptr || N == 0, "V is NULL");
    mpb200_samples *s = new (std::nothrow) mpb200_samples();
    if (!s) return fail(MPB200_ENOMEM, "out of host memory");
    s->N = N;
    s->d = d;
    s->q0 = 0;
    s->q1 = N;
    int rc = s->V.reserve(sizeof(double) * (size_t)(N * d + 1));
    if (rc) { delete s; return rc; }
    if (N > 0) {
        cudaError_t e = cudaMemcpyAsync(s->V.p, V_aos, sizeof(double) * (size_t)(N * d), cudaMemcpyHostToDevice, ctx().stream);
        if (e != cudaSuccess) { s->V.release(); delete s; return fail(MPB200_ECUDA, "H2D copy failed: %s", cudaGetErrorString(e)); }
    }
    rc = finish_samples(s);
    if (rc) { mpb200_samples_destroy(s); return rc; }
    *out = s;
    return MPB200_OK;
}
int mpb200_sample_free(const mpb200_obstacles *o, const mpb200_space_desc *ss, int64_t N, uint64_t seed, int32_t order,
                       mpb200_samples **out, double *V_host, int64_t *candidates) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(o != nullptr && ss != nullptr && out != nullptr, "NULL argument");
    MPB_CHECK_ARG(N >= 0 && N < INT_MAX, "N out of range");
    MPB_CHECK_ARG(ss->n >= 1 && ss->n <= kMaxDim, "state dimension out of range (1..16)");
    MPB_CHECK_ARG(order == MPB200_ORDER_CANDIDATE || order == MPB200_ORDER_MORTON, "order must be 0 (candidate) or 1 (Morton)");
    mpb200_samples *s = new (std::nothrow) mpb200_samples();
    if (!s) return fail(MPB200_ENOMEM, "out of host memory");
    s->N = N;
    s->d = ss->n;
    s->q0 = 0;
    s->q1 = N;
    int rc = s->V.reserve(sizeof(double) * (size_t)(N * s->d + 1));
    int64_t used = 0;
    if (!rc && N > 0) rc = sample_free_device(o, ss, N, seed, s->V.as<double>(), s->q_order, s->scan_tmp, &used);
    if (!rc && order == MPB200_ORDER_MORTON) rc = morton_reorder_device(s->V.as<double>(), N, ss, s->q_order);
    if (!rc) rc = finish_samples(s);
    if (!rc && V_host && N > 0) {
        cudaStream_t st = ctx().stream;
        cudaError_t e = cudaMemcpyAsync(V_host, s->V.p, sizeof(double) * (size_t)(N * s->d), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) rc = fail(MPB200_ECUDA, "D2H copy failed: %s", cudaGetErrorString(e));
    }
    if (rc) { mpb200_samples_destroy(s); return rc; }
    if (candidates) *candidates = used;
    *out = s;
    return MPB200_OK;
}
int mpb200_samples_destroy(mpb200_samples *s) {
    if (!s) return MPB200_OK;
    if (ctx().ready) cudaStreamSynchronize(ctx().stream);
    if (s->graph_exec) cudaGraphExecDestroy(s->graph_exec);
    if (s->shadow_xy) mpb200_samples_destroy(s->shadow_xy);
    if (s->shadow_cand) mpb200_table_destroy(s->shadow_cand);
    s->car_work.release();
    s->V.release(); s->cell_start.release(); s->cell_fill.release(); s->sorted_idx.release();
    s->sorted_pos.release(); s->pt_order.release(); s->minmax.release(); s->scan_tmp.release(); s->point_bits.release(); s->q_order.release(); s->aux.release();
    delete s;
    return MPB200_OK;
}
int mpb200_samples_set_query_range(mpb200_samples *s, int64_t q0, int64_t q1) {
    MPB_CHECK_ARG(s != nullptr, "samples handle is NULL");
    MPB_CHECK_ARG(0 <= q0 && q0 <= q1 && q1 <= s->N, "query range must satisfy 0 <= q0 <= q1 <= N");
    s->q0 = q0;
    s->q1 = q1;
    s->pt_order_valid = false;
    // bounding box of the shard's own samples: the grid only has to cover it (+ r)
    memcpy(s->h_qbbox, s->h_bbox, sizeof(s->h_bbox));
    if (ctx().ready && q1 > q0 && (q0 != 0 || q1 != s->N)) {
        cudaStream_t st = ctx().stream;
        if (int rc = compute_bbox(s, q0, q1)) return rc;
        MPB_CUDA(cudaMemcpyAsync(s->h_qbbox, s->minmax.p, sizeof(double) * 2 * s->d, cudaMemcpyDeviceToHost, st));
        MPB_CUDA(cudaStreamSynchronize(st));
    }
    return MPB200_OK;
}

// ---- Euclidean r-ball table -----------------------------------------------------------
int mpb200_inball_build(mpb200_samples *s, double r, mpb200_table **table, int64_t *nnz) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(s != nullptr && table != nullptr, "NULL handle");
    MPB_CHECK_ARG(r >= 0 && r == r, "r must be a non-negative number");
    mpb200_table *t = *table;
    bool fresh = false;
    if (!t) {
        t = new (std::nothrow) mpb200_table();
        if (!t) return fail(MPB200_ENOMEM, "out of host memory");
        fresh = true;
    }
    t->edge_bits_valid = false;  // bits of an earlier build do not describe the new table
    t->src_N = s->N;
    t->src_d = s->d;
    t->src_serial = s->serial;
    int rc;
    if (s->N == 0) {
        rc = t->colptr.reserve(sizeof(int64_t));
        if (!rc) {
            int64_t one = 1;
            rc = upload_sync(t->colptr.p, &one, sizeof(one));
            t->ncols = 0; t->col0 = 0; t->nnz = 0; t->r = r; t->euclid = true; t->has_order = false;
        }
    } else if (s->d <= 3 && s->d >= 2) {
        rc = grid_inball_build(s, r, t);
    } else {
        rc = brute_inball_build(s, r, t);
    }
    if (rc) {
        if (fresh) mpb200_table_destroy(t);
        return rc;
    }
    *table = t;
    if (nnz) *nnz = t->nnz;
    return MPB200_OK;
}
int mpb200_inball_build_checked(mpb200_samples *s, double r, const mpb200_obstacles *o, const mpb200_space_desc *ss,
                                mpb200_table **table, int64_t *nnz, int64_t *checks) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(s != nullptr && table != nullptr && o != nullptr && ss != nullptr, "NULL handle");
    MPB_CHECK_ARG(r >= 0 && r == r, "r must be a non-negative number");
    if (int rc = mpb200_inball_build(s, r, table, nnz)) return rc;
    return mpb200_edges_free(s, *table, o, ss, nullptr, checks);
}
int mpb200_table_fetch_edge_bits(const mpb200_table *t, uint64_t *bitchunks) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(t != nullptr && bitchunks != nullptr, "NULL argument");
    if (t->nnz > 0 && !(t->edge_bits_valid && t->edge_bits_nnz == t->nnz))
        return fail(MPB200_ESTATE, "no edge validity has been computed for the current contents of this table");
    const size_t words = (size_t)ceil_div(t->nnz, 64);
    cudaStream_t st = ctx().stream;
    if (words) MPB_CUDA(cudaMemcpyAsync(bitchunks, t->edge_bits.p, sizeof(uint64_t) * words, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    return MPB200_OK;
}
int mpb200_table_nnz(const mpb200_table *t, int64_t *nnz, int64_t *ncols) {
    MPB_CHECK_ARG(t != nullptr, "table handle is NULL");
    if (nnz) *nnz = t->nnz;
    if (ncols) *ncols = t->ncols;
    return MPB200_OK;
}
int mpb200_table_device_view(const mpb200_table *t, void **colptr, void **rowval, void **nzval, void **edge_bits) {
    MPB_CHECK_ARG(t != nullptr, "table handle is NULL");
    if (colptr) *colptr = t->colptr.p;
    if (rowval) *rowval = t->rowval.p;
    if (nzval) *nzval = t->nzval.p;
    if (edge_bits) *edge_bits = (t->edge_bits_valid && t->edge_bits_nnz == t->nnz) ? t->edge_bits.p : nullptr;  // never stale bits
    return MPB200_OK;
}
// ---- table fetch -----------------------------------------------------------------------------------------
// The reference's table format (Int64 rowval + Float64 nzval, 16 bytes per stored neighbour) makes the fetch
// PCIe-bound: 27.5M entries = 441 MB = 7.9 ms at 57 GB/s against 0.56 ms of kernels.  The row indices are sample
// numbers <= N, so they cross the bus bit-packed -- B = the smallest multiple of 4 bits that holds N (20 bits for
// N = 1M; eight indices fill exactly B/4 32-bit words) -- packed on the device into pinned staging in chunks, and are
// unpacked into the caller's Int64 array by a few host threads WHILE the nzval transfer is still running:
// fewer bytes on the wire (8 -> 2.5 bytes per index at N = 1M), the same bytes in the caller's arrays.
}  // extern "C"
namespace fetchd {
template <int BITS>
__global__ void __launch_bounds__(256) pack_rows_kernel(const int64_t *__restrict__ in, int64_t n, int64_t groups,
                                                        uint32_t *__restrict__ out) {
    constexpr int W = BITS / 4;  // words per group of eight indices
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += (int64_t)gridDim.x * blockDim.x) {
        unsigned long long acc = 0;
        int nb = 0, w = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int64_t e = 8 * g + i;
            const unsigned long long v = e < n ? (unsigned long long)in[e] : 0ULL;
            acc |= v << nb;
            nb += BITS;
            if (nb >= 32) {
                out[g * W + w++] = (uint32_t)acc;
                acc >>= 32;
                nb -= 32;
            }
        }
    }
}
// host side of the same format: groups [g0, g1) of `in` -> dst[8 g0 .. min(8 g1, n)), streaming stores
template <int BITS>
static void unpack_rows(const uint32_t *in, int64_t g0, int64_t g1, int64_t n, long long *dst) {
    constexpr int W = BITS / 4;
    constexpr unsigned long long mask = BITS == 32 ? 0xffffffffULL : ((1ULL << BITS) - 1ULL);
    for (int64_t g = g0; g < g1; ++g) {
        const uint32_t *p = in + g * W;
        unsigned long long acc = 0;
        int nb = 0, w = 0;
        const int64_t base = 8 * g;
        const int lim = (int)std::min<int64_t>(8, n - base);
        for (int i = 0; i < lim; ++i) {
            if (nb < BITS) {
                acc |= (unsigned long long)p[w++] << nb;
                nb += 32;
            }
            _mm_stream_si64(dst + base + i, (long long)(acc & mask));
            acc >>= BITS;
            nb -= BITS;
        }
    }
    _mm_sfence();
}
constexpr int kFetchChunks = 32;
void *g_pin = nullptr;  // pinned staging for the packed indices (library-owned, grows, reused)
size_t g_pin_cap = 0;
cudaEvent_t g_fetch_ev[kFetchChunks] = {};
}  // namespace fetchd
using namespace fetchd;

static int index_bits(int64_t max_value) {
    int b = 1;
    while (b < 32 && (int64_t(1) << b) <= max_value) ++b;
    b = (b + 3) & ~3;
    return b < 12 ? 12 : b;
}

static int fetch_rows_narrow(mpb200_table *t, int64_t *rowval, cudaStream_t st, std::vector<std::thread> *workers) {
    const int64_t nnz = t->nnz;
    static const int env_bits = [] { const char *e = getenv("MPB200_FETCH_BITS"); return e ? atoi(e) : 0; }();
    const int bits = (env_bits >= 12 && env_bits <= 32 && env_bits % 4 == 0) ? env_bits
                     : (t->src_N > 0 ? index_bits(t->src_N) : 32);
    if (t->src_N > 0 && bits < 32 && (int64_t(1) << bits) <= t->src_N) return 1;  // a forced width that cannot hold N
    const int W = bits / 4;
    const int64_t groups = ceil_div(nnz, 8);
    const size_t bytes = sizeof(uint32_t) * (size_t)groups * (size_t)W;
    if (int rc = t->scratch.reserve(bytes)) return rc;
    if (g_pin_cap < bytes) {
        if (g_pin) cudaFreeHost(g_pin);
        g_pin = nullptr;
        g_pin_cap = bytes + bytes / 8;
        if (cudaMallocHost(&g_pin, g_pin_cap) != cudaSuccess) {
            cudaGetLastError();
            g_pin = nullptr;
            g_pin_cap = 0;
            return 1;  // no staging: the caller falls back to the plain copy
        }
    }
    for (int k = 0; k < kFetchChunks; ++k)
        if (!g_fetch_ev[k]) MPB_CUDA(cudaEventCreateWithFlags(&g_fetch_ev[k], cudaEventDisableTiming));
    uint32_t *d32 = t->scratch.as<uint32_t>();
    uint32_t *h32 = static_cast<uint32_t *>(g_pin);
    const unsigned grid = (unsigned)(ctx().sm_count * 8);
    const int64_t *src = t->rowval.as<int64_t>();
    switch (bits) {
        case 12: pack_rows_kernel<12><<<grid, 256, 0, st>>>(src, nnz, groups, d32); break;
        case 16: pack_rows_kernel<16><<<grid, 256, 0, st>>>(src, nnz, groups, d32); break;
        case 20: pack_rows_kernel<20><<<grid, 256, 0, st>>>(src, nnz, groups, d32); break;
        case 24: pack_rows_kernel<24><<<grid, 256, 0, st>>>(src, nnz, groups, d32); break;
        case 28: pack_rows_kernel<28><<<grid, 256, 0, st>>>(src, nnz, groups, d32); break;
        default: pack_rows_kernel<32><<<grid, 256, 0, st>>>(src, nnz, groups, d32); break;
    }
    MPB_LAUNCHED();
    const int64_t per = ceil_div(groups, kFetchChunks);  // groups per chunk
    for (int k = 0; k < kFetchChunks; ++k) {
        const int64_t a = std::min<int64_t>(k * per, groups), b = std::min<int64_t>(a + per, groups);
        if (b > a)
            MPB_CUDA(cudaMemcpyAsync(h32 + a * W, d32 + a * W, sizeof(uint32_t) * (size_t)((b - a) * W), cudaMemcpyDeviceToHost, st));
        MPB_CUDA(cudaEventRecord(g_fetch_ev[k], st));
    }
    // unpacking threads: chunk k is converted as soon as its copy has landed (the nzval copy queued behind keeps the
    // bus busy); streaming stores: the destination is written once and not read here (no read-for-ownership traffic
    // on a memory bus that is taking the nzval DMA at the same time)
    const int device = ctx().device;
    static const int env_threads = [] { const char *e = getenv("MPB200_FETCH_THREADS"); return e ? atoi(e) : 0; }();
    // default: up to 8 threads, but no more than this process's share of the host cores when several ranks share the
    // box (torchrun exports LOCAL_WORLD_SIZE): oversubscribed unpacking threads cost more than they give
    static const unsigned local_world = [] { const char *e = getenv("LOCAL_WORLD_SIZE"); const int v = e ? atoi(e) : 1; return (unsigned)(v > 0 ? v : 1); }();
    const int nthreads = env_threads > 0 ? std::min(env_threads, kFetchChunks)
                                         : (int)std::max(1u, std::min(8u, std::thread::hardware_concurrency() / local_world));
    for (int w = 0; w < nthreads; ++w)
        workers->emplace_back([=]() {
            cudaSetDevice(device);
            long long *dst = reinterpret_cast<long long *>(rowval);
            for (int k = w; k < kFetchChunks; k += nthreads) {
                cudaEventSynchronize(g_fetch_ev[k]);
                const int64_t a = std::min<int64_t>(k * per, groups), b = std::min<int64_t>(a + per, groups);
                switch (bits) {
                    case 12: unpack_rows<12>(h32, a, b, nnz, dst); break;
                    case 16: unpack_rows<16>(h32, a, b, nnz, dst); break;
                    case 20: unpack_rows<20>(h32, a, b, nnz, dst); break;
                    case 24: unpack_rows<24>(h32, a, b, nnz, dst); break;
                    case 28: unpack_rows<28>(h32, a, b, nnz, dst); break;
                    default: unpack_rows<32>(h32, a, b, nnz, dst); break;
                }
            }
        });
    return 0;
}

extern "C" {
int mpb200_table_fetch(const mpb200_table *t_, int64_t *colptr, int64_t *rowval, double *nzval) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(t_ != nullptr, "table handle is NULL");
    mpb200_table *t = const_cast<mpb200_table *>(t_);
    cudaStream_t st = ctx().stream;
    static const bool plain = getenv("MPB200_FETCH_PLAIN") != nullptr;
    std::vector<std::thread> workers;
    bool narrowed = false;
    int rc = 0;
    if (rowval && t->nnz >= (int64_t(1) << 20) && !plain) {  // below ~1M entries the plain copy is already sub-millisecond
        rc = fetch_rows_narrow(t, rowval, st, &workers);
        narrowed = rc == 0;
        if (rc < 0) {  // a CUDA error inside: collect the threads already started before reporting it
            for (auto &w : workers) w.join();
            return rc;
        }
        rc = 0;
    }
    cudaError_t e = cudaSuccess;
    if (rowval && t->nnz && !narrowed)
        e = cudaMemcpyAsync(rowval, t->rowval.p, sizeof(int64_t) * (size_t)t->nnz, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && nzval && t->nnz)
        e = cudaMemcpyAsync(nzval, t->nzval.p, sizeof(double) * (size_t)t->nnz, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && colptr)
        e = cudaMemcpyAsync(colptr, t->colptr.p, sizeof(int64_t) * (size_t)(t->ncols + 1), cudaMemcpyDeviceToHost, st);
    for (auto &w : workers) w.join();
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail(MPB200_ECUDA, "table fetch failed: %s", cudaGetErrorString(e));
    return MPB200_OK;
}
}  // extern "C"
static void release_fetch_staging() {
    if (g_pin) cudaFreeHost(g_pin);
    g_pin = nullptr;
    g_pin_cap = 0;
    for (int k = 0; k < kFetchChunks; ++k)
        if (g_fetch_ev[k]) cudaEventDestroy(g_fetch_ev[k]), g_fetch_ev[k] = nullptr;
}
extern "C" {
int mpb200_table_destroy(mpb200_table *t) {
    if (!t) return MPB200_OK;
    if (ctx().ready) cudaStreamSynchronize(ctx().stream);
    t->colptr.release(); t->rowval.release(); t->nzval.release(); t->counts.release(); t->masks.release();
    t->edge_bits.release(); t->scratch.release(); t->col_list.release(); t->col_order.release();
    delete t;
    return MPB200_OK;
}

// ---- obstacles ----------------------------------------------------------------------------
int mpb200_obstacles2d_create(const mpb200_obstacles2d_desc *d, mpb200_obstacles **out) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(d != nullptr && out != nullptr, "NULL argument");
    MPB_CHECK_ARG(d->n_gates >= 0 && d->n_gates <= kMaxGates, "too many compound gates (max 32)");
    MPB_CHECK_ARG(d->n_shapes >= 0, "negative shape count");
    MPB_CHECK_ARG(d->n_shapes == 0 || (d->shape_kind && d->shape_gate && d->shape_off && d->data), "NULL shape arrays");
    MPB_CHECK_ARG(d->n_gates == 0 || (d->gate_parent && d->gate_aabb), "NULL gate arrays");
    const int G = d->n_gates, S = d->n_shapes;
    const int data_words = S ? d->shape_off[S] : 0;
    // layout (predicates.cuh): int directory | gate AABBs | shape data
    const int dir_words = (4 + G + 4 * S + 1) / 2;
    const int gate_base = dir_words;
    const int cull_base = gate_base + 4 * G;
    const int base = cull_base + 4 * S;
    std::vector<double> T((size_t)(base + data_words + 1), 0.0);
    int *I = reinterpret_cast<int *>(T.data());
    I[0] = G; I[1] = S; I[2] = d->flags; I[3] = gate_base;
    for (int g = 0; g < G; ++g) {
        MPB_CHECK_ARG(d->gate_parent[g] < g && d->gate_parent[g] >= -1, "gate parents must precede their children");
        I[4 + g] = d->gate_parent[g];
        for (int k = 0; k < 4; ++k) T[gate_base + 4 * g + k] = d->gate_aabb[4 * g + k];
    }
    for (int s = 0; s < S; ++s) {
        int len = d->shape_off[s + 1] - d->shape_off[s];
        int kind = d->shape_kind[s];
        MPB_CHECK_ARG(kind == 0 || kind == 1, "shape_kind must be 0 (Circle) or 1 (Polygon)");
        MPB_CHECK_ARG(d->shape_gate[s] >= -1 && d->shape_gate[s] < G, "shape_gate out of range");
        int K = 0;
        if (kind == 0) {
            MPB_CHECK_ARG(len == 7, "Circle record must have 7 doubles");
            MPB_CHECK_ARG(d->data[d->shape_off[s] + 2] > 0, "Radius must be positive");  // SAT2D.jl:19
        } else {
            MPB_CHECK_ARG(len >= 4 + 18 && (len - 4) % 6 == 0, "Polygon record must have 4+6K doubles, K >= 3");  // SAT2D.jl:39
            K = (len - 4) / 6;
        }
        int *dir = I + 4 + G + 4 * s;
        dir[0] = kind; dir[1] = d->shape_gate[s]; dir[2] = base + d->shape_off[s]; dir[3] = K;
    }
    for (int i = 0; i < data_words; ++i) T[base + i] = d->data[i];
    // cull boxes + gate consistency (predicates.cuh): AABB of shape s inside its gate chain
    auto inside = [](const double *in, const double *out) {
        return out[0] <= in[0] && in[1] <= out[1] && out[2] <= in[2] && in[3] <= out[3];
    };
    bool consistent = true;
    for (int g = 0; g < G; ++g)
        if (d->gate_parent[g] >= 0 && !inside(&d->gate_aabb[4 * g], &d->gate_aabb[4 * d->gate_parent[g]])) consistent = false;
    for (int s = 0; s < S; ++s) {
        const double *rec = d->data + d->shape_off[s];
        const double *own = d->shape_kind[s] == 0 ? rec + 3 : rec;  // xlo xhi ylo yhi
        if (d->shape_gate[s] >= 0 && !inside(own, &d->gate_aabb[4 * d->shape_gate[s]])) consistent = false;
    }
    const double inf = std::numeric_limits<double>::infinity();
    for (int s = 0; s < S; ++s) {
        double *cb = &T[cull_base + 4 * s];
        const double *rec = d->data + d->shape_off[s];
        if (!consistent || (d->shape_kind[s] == 0 && d->shape_gate[s] < 0)) {
            cb[0] = -inf; cb[1] = inf; cb[2] = -inf; cb[3] = inf;
        } else if (d->shape_kind[s] == 0) {
            for (int k = 0; k < 4; ++k) cb[k] = d->gate_aabb[4 * d->shape_gate[s] + k];
        } else {
            for (int k = 0; k < 4; ++k) cb[k] = rec[k];
        }
    }
    if (consistent) I[2] |= 2;
    mpb200_obstacles *o = new (std::nothrow) mpb200_obstacles();
    if (!o) return fail(MPB200_ENOMEM, "out of host memory");
    o->kind = 0; o->n_gates = G; o->n_shapes = S; o->flags = d->flags;
    o->table_words = base + data_words;
    o->M = 0; o->d = 2;
    int rc = o->table.reserve(sizeof(double) * T.size());
    if (!rc) rc = upload_sync(o->table.p, T.data(), sizeof(double) * T.size());
    if (rc) { o->table.release(); delete o; return rc; }
    *out = o;
    return MPB200_OK;
}
int mpb200_boxes_create(const double *lo, const double *hi, int M, int d, mpb200_obstacles **out) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(out != nullptr, "out is NULL");
    MPB_CHECK_ARG(M >= 0 && d >= 1 && d <= kMaxDim, "bad box count / dimension");
    MPB_CHECK_ARG(M == 0 || (lo && hi), "NULL box arrays");
    std::vector<double> T((size_t)(2 * M * d + 1), 0.0);
    for (int i = 0; i < M * d; ++i) { T[i] = lo[i]; T[(size_t)M * d + i] = hi[i]; }
    mpb200_obstacles *o = new (std::nothrow) mpb200_obstacles();
    if (!o) return fail(MPB200_ENOMEM, "out of host memory");
    o->kind = 1; o->M = M; o->d = d; o->table_words = 2 * M * d;
    int rc = o->table.reserve(sizeof(double) * T.size());
    if (!rc) rc = upload_sync(o->table.p, T.data(), sizeof(double) * T.size());
    if (rc) { o->table.release(); delete o; return rc; }
    *out = o;
    return MPB200_OK;
}
int mpb200_obstacles_destroy(mpb200_obstacles *o) {
    if (!o) return MPB200_OK;
    if (ctx().ready) cudaStreamSynchronize(ctx().stream);
    o->table.release();
    delete o;
    return MPB200_OK;
}

// ---- batched validity ------------------------------------------------------------------------
int mpb200_points_free(const mpb200_samples *s_, const mpb200_obstacles *o, const mpb200_space_desc *ss,
                       uint64_t *bitchunks) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(s_ != nullptr, "samples handle is NULL");
    mpb200_samples *s = const_cast<mpb200_samples *>(s_);
    cudaStream_t st = ctx().stream;
    const int64_t n = s->q1 - s->q0;  // this process's shard of the samples (all of them by default)
    const size_t words = (size_t)ceil_div(n, 64);
    s->point_bits_valid = false;
    if (int rc = s->point_bits.reserve(sizeof(uint64_t) * (words + 1))) return rc;
    phase_bank(MPB200_OP_POINTS);
    phase_mark(0);
    MPB_CUDA(cudaMemsetAsync(s->point_bits.p, 0, sizeof(uint64_t) * (words + 1), st));
    // after a grid build the samples are visited in cell order: neighbouring lanes test neighbouring points
    if (int rc = points_free_device(s->V.as<double>() + s->q0 * s->d, n, s->d, o, ss, s->point_bits.as<uint32_t>(), nullptr, s))
        return rc;
    s->point_bits_valid = s->q0 == 0 && s->q1 == s->N;
    phase_mark(1);
    phases_collect(1);
    if (bitchunks) {  // NULL: asynchronous, the bits stay on the device (stream-ordered with later calls)
        if (words) MPB_CUDA(cudaMemcpyAsync(bitchunks, s->point_bits.p, sizeof(uint64_t) * words, cudaMemcpyDeviceToHost, st));
        MPB_CUDA(cudaStreamSynchronize(st));
    }
    return MPB200_OK;
}

int mpb200_edges_free(const mpb200_samples *s, const mpb200_table *t_, const mpb200_obstacles *o,
                      const mpb200_space_desc *ss, uint64_t *bitchunks, int64_t *checks) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(s != nullptr && t_ != nullptr, "NULL handle");
    mpb200_table *t = const_cast<mpb200_table *>(t_);
    MPB_CHECK_ARG(t->src_N == s->N && t->src_d == s->d, "the table was not built from this sample set");
    Context &c = ctx();
    cudaStream_t st = c.stream;
    const size_t words = (size_t)ceil_div(t->nnz, 64);
    // the bits, one spare word, then the pass's counters (segment tests run, columns left for the per-edge test):
    // one memset clears them all
    if (int rc = t->edge_bits.reserve(sizeof(uint64_t) * (words + 3))) return rc;
    unsigned long long *d_counters = t->edge_bits.as<unsigned long long>() + words + 1;
    t->edge_bits_valid = false;
    phase_bank(MPB200_OP_EDGES);
    phase_mark(0);
    MPB_CUDA(cudaMemsetAsync(t->edge_bits.p, 0, sizeof(uint64_t) * (words + 3), st));
    if (int rc = edges_free_device(s, t, o, ss, t->edge_bits.as<uint32_t>(), d_counters))
        return rc;
    t->edge_bits_valid = true;
    t->edge_bits_nnz = t->nnz;
    phase_mark(1);
    phases_collect(1);
    if (bitchunks || checks) {  // both NULL: asynchronous, the bits stay on the device
        if (bitchunks && words)
            MPB_CUDA(cudaMemcpyAsync(bitchunks, t->edge_bits.p, sizeof(uint64_t) * words, cudaMemcpyDeviceToHost, st));
        MPB_CUDA(cudaMemcpyAsync(c.h_scalar + 4, d_counters, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        MPB_CUDA(cudaStreamSynchronize(st));
        if (checks) *checks = c.h_scalar[4];
    }
    return MPB200_OK;
}

static int batch_states(const double *v, const double *w, int64_t n, int d, const mpb200_obstacles *o,
                        const mpb200_space_desc *ss, uint8_t *out) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(n >= 0 && d >= 1 && d <= kMaxDim, "bad batch size / dimension");
    MPB_CHECK_ARG(n == 0 || (v && out), "NULL buffers");
    if (n == 0) return MPB200_OK;
    cudaStream_t st = ctx().stream;
    static DevBuf bufA, bufB, bufO;  // reused staging (single caller thread, see DESIGN.md threading)
    size_t bytes = sizeof(double) * (size_t)(n * d);
    if (int rc = bufA.reserve(bytes)) return rc;
    if (int rc = bufO.reserve((size_t)n + 64)) return rc;
    MPB_CUDA(cudaMemcpyAsync(bufA.p, v, bytes, cudaMemcpyHostToDevice, st));
    int rc;
    if (w) {
        if ((rc = bufB.reserve(bytes))) return rc;
        MPB_CUDA(cudaMemcpyAsync(bufB.p, w, bytes, cudaMemcpyHostToDevice, st));
        rc = segments_free_device(bufA.as<double>(), bufB.as<double>(), n, d, o, ss, bufO.as<uint8_t>());
    } else {
        rc = points_free_device(bufA.as<double>(), n, d, o, ss, nullptr, bufO.as<uint8_t>());
    }
    if (rc) return rc;
    MPB_CUDA(cudaMemcpyAsync(out, bufO.p, (size_t)n, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    return MPB200_OK;
}
int mpb200_states_free(const double *v_aos, int64_t n, int d, const mpb200_obstacles *o, const mpb200_space_desc *ss,
                       uint8_t *out) {
    return batch_states(v_aos, nullptr, n, d, o, ss, out);
}
int mpb200_segments_free(const double *v_aos, const double *w_aos, int64_t n, int d, const mpb200_obstacles *o,
                         const mpb200_space_desc *ss, uint8_t *out) {
    MPB_CHECK_ARG(n == 0 || w_aos != nullptr, "w is NULL");
    return batch_states(v_aos, w_aos, n, d, o, ss, out);
}

// ---- linear-quadratic steering --------------------------------------------------------------------
int mpb200_lq_create(const double *A, const double *B, const double *c, const double *R, int n, int m, mpb200_lq **out) {
    MPB_CHECK_ARG(A && B && c && R && out, "NULL argument");
    MPB_CHECK_ARG(n >= 1 && n <= kLqgMaxN && m >= 1 && m <= kLqgMaxN, "state / control dimension out of range (1..6)");
    for (int i = 0; i < m; ++i)
        for (int j = 0; j < m; ++j) MPB_CHECK_ARG(R[i + j * m] == R[j + i * m], "R must be symmetric");
    // the double-integrator family (linearquadratic.jl:46-53: A = [0 I; 0 0], B = [0; I], c = 0, m = 1..3) keeps its
    // closed form and the two-stage kernel of lq.cu; every other nilpotent (A, B, c) takes the numeric path
    bool di = (n == 2 * m) && m <= 3;
    for (int j = 0; di && j < n; ++j)
        for (int i = 0; i < n; ++i) di = di && (A[i + j * n] == ((j == i + m) ? 1.0 : 0.0));
    for (int j = 0; di && j < m; ++j)
        for (int i = 0; i < n; ++i) di = di && (B[i + j * n] == ((i == j + m) ? 1.0 : 0.0));
    for (int i = 0; di && i < n; ++i) di = di && (c[i] == 0.0);
    mpb200_lq *lq = new (std::nothrow) mpb200_lq();
    if (!lq) return fail(MPB200_ENOMEM, "out of host memory");
    if (di) {
        bool scalar = true;
        for (int i = 0; i < m; ++i)
            for (int j = 0; j < m; ++j) {
                if (i != j && R[i + j * m] != 0.0) scalar = false;
                if (i == j && R[i + j * m] != R[0]) scalar = false;
            }
        for (int i = 0; i < m; ++i)
            if (!(R[i + i * m] > 0.0)) { delete lq; return fail(MPB200_EARG, "R must be positive definite"); }
        lq->d = m;
        lq->scalar_R = scalar;
        for (int i = 0; i < m; ++i)
            for (int j = 0; j < m; ++j) lq->R[i * m + j] = R[i + j * m];
    } else {
        MPB_REQUIRE_INIT();
        // column-major (Julia) -> row-major tables; expAt's nilpotency check (linearquadratic.jl:94-98) is inside
        double Ar[kLqgMaxN * kLqgMaxN], Br[kLqgMaxN * kLqgMaxN], Rr[kLqgMaxN * kLqgMaxN];
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j) Ar[i * n + j] = A[i + j * n];
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < m; ++j) Br[i * m + j] = B[i + j * n];
        for (int i = 0; i < m; ++i)
            for (int j = 0; j < m; ++j) Rr[i * m + j] = R[i + j * m];
        lq->general = true;
        int rc = lqg_setup_host(n, m, Ar, Br, c, Rr, &lq->gen);
        if (!rc) rc = lqg_upload(lq);
        if (rc) { lq->gen_dev.release(); delete lq; return rc; }
    }
    *out = lq;
    return MPB200_OK;
}
int mpb200_lq_destroy(mpb200_lq *lq) {
    if (!lq) return MPB200_OK;
    if (ctx().ready) cudaStreamSynchronize(ctx().stream);
    lq->gen_dev.release();
    delete lq;
    return MPB200_OK;
}

int mpb200_lq_inball_build(mpb200_samples *s, const mpb200_lq *lq, double r, mpb200_table **tableF, mpb200_table **tableB,
                           int64_t *nnzF, int64_t *nnzB) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(s && lq && tableF && tableB, "NULL handle");
    MPB_CHECK_ARG(r > 0 && r == r, "r must be positive");
    mpb200_table *tF = *tableF, *tB = *tableB;
    const bool freshF = !tF, freshB = !tB;
    if (!tF) tF = new (std::nothrow) mpb200_table();
    if (!tB) tB = new (std::nothrow) mpb200_table();
    if (!tF || !tB) return fail(MPB200_ENOMEM, "out of host memory");
    tF->edge_bits_valid = tB->edge_bits_valid = false;
    tF->src_N = tB->src_N = s->N;
    tF->src_d = tB->src_d = s->d;
    tF->src_serial = tB->src_serial = s->serial;
    int rc = lq->general ? lqg_inball_build(s, lq, r, tF, tB) : lq_inball_build(s, lq, r, tF, tB);
    if (rc) {
        if (freshF) mpb200_table_destroy(tF);
        if (freshB) mpb200_table_destroy(tB);
        return rc;
    }
    *tableF = tF;
    *tableB = tB;
    if (nnzF) *nnzF = tF->nnz;
    if (nnzB) *nnzB = tB->nnz;
    return MPB200_OK;
}

int mpb200_lq_steer(const mpb200_lq *lq, const double *v, const double *w, int64_t n, double r, double *cost,
                    double *topt) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(lq && (n == 0 || (v && w && cost && topt)), "NULL argument");
    if (n == 0) return MPB200_OK;
    cudaStream_t st = ctx().stream;
    static DevBuf bufA, bufB, bufC, bufT;
    const int ns = lq->general ? lq->gen.n : 2 * lq->d;
    const size_t bytes = sizeof(double) * (size_t)(n * ns);
    if (int rc = bufA.reserve(bytes)) return rc;
    if (int rc = bufB.reserve(bytes)) return rc;
    if (int rc = bufC.reserve(sizeof(double) * (size_t)n)) return rc;
    if (int rc = bufT.reserve(sizeof(double) * (size_t)n)) return rc;
    MPB_CUDA(cudaMemcpyAsync(bufA.p, v, bytes, cudaMemcpyHostToDevice, st));
    MPB_CUDA(cudaMemcpyAsync(bufB.p, w, bytes, cudaMemcpyHostToDevice, st));
    if (int rc = (lq->general ? lqg_steer_device : lq_steer_device)(lq, bufA.as<double>(), bufB.as<double>(), n, r,
                                                                    bufC.as<double>(), bufT.as<double>()))
        return rc;
    MPB_CUDA(cudaMemcpyAsync(cost, bufC.p, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaMemcpyAsync(topt, bufT.p, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    return MPB200_OK;
}

int mpb200_lq_edges_free(const mpb200_samples *s, const mpb200_table *t_, const mpb200_lq *lq, double r,
                         const mpb200_obstacles *o, const mpb200_space_desc *ss, uint64_t *bitchunks, int64_t *checks) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(s && t_ && lq && o, "NULL handle");
    mpb200_table *t = const_cast<mpb200_table *>(t_);
    MPB_CHECK_ARG(t->src_N == s->N && t->src_d == s->d, "the table was not built from this sample set");
    Context &c = ctx();
    cudaStream_t st = c.stream;
    const size_t words = (size_t)ceil_div(t->nnz, 64);
    if (int rc = t->edge_bits.reserve(sizeof(uint64_t) * (words + 1))) return rc;
    t->edge_bits_valid = false;
    phase_bank(MPB200_OP_EDGES);
    phase_mark(0);
    MPB_CUDA(cudaMemsetAsync(t->edge_bits.p, 0, sizeof(uint64_t) * (words + 1), st));
    MPB_CUDA(cudaMemsetAsync(c.d_scalar + 4, 0, sizeof(int64_t), st));
    if (int rc = (lq->general ? lqg_edges_free_device : lq_edges_free_device)(
            s, t, lq, r, o, ss, t->edge_bits.as<uint32_t>(), reinterpret_cast<unsigned long long *>(c.d_scalar + 4)))
        return rc;
    t->edge_bits_valid = true;
    t->edge_bits_nnz = t->nnz;
    phase_mark(1);
    phases_collect(1);
    if (bitchunks || checks) {  // both NULL: asynchronous, the bits stay on the device
        if (bitchunks && words)
            MPB_CUDA(cudaMemcpyAsync(bitchunks, t->edge_bits.p, sizeof(uint64_t) * words, cudaMemcpyDeviceToHost, st));
        MPB_CUDA(cudaMemcpyAsync(c.h_scalar + 4, c.d_scalar + 4, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        MPB_CUDA(cudaStreamSynchronize(st));
        if (checks) *checks = c.h_scalar[4];
    }
    return MPB200_OK;
}

int mpb200_lq_motions_free(const mpb200_lq *lq, double r, const double *v, const double *w, int64_t n,
                           const mpb200_obstacles *o, const mpb200_space_desc *ss, uint8_t *out, int64_t *checks) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(lq && o && (n == 0 || (v && w && out)), "NULL argument");
    if (checks) *checks = 0;
    if (n == 0) return MPB200_OK;
    Context &c = ctx();
    cudaStream_t st = c.stream;
    static DevBuf bufA, bufB, bufO;
    const int ns = lq->general ? lq->gen.n : 2 * lq->d;
    const size_t bytes = sizeof(double) * (size_t)(n * ns);
    if (int rc = bufA.reserve(bytes)) return rc;
    if (int rc = bufB.reserve(bytes)) return rc;
    if (int rc = bufO.reserve((size_t)n + 64)) return rc;
    MPB_CUDA(cudaMemcpyAsync(bufA.p, v, bytes, cudaMemcpyHostToDevice, st));
    MPB_CUDA(cudaMemcpyAsync(bufB.p, w, bytes, cudaMemcpyHostToDevice, st));
    MPB_CUDA(cudaMemsetAsync(c.d_scalar + 5, 0, sizeof(int64_t), st));
    if (int rc = (lq->general ? lqg_motions_free_device : lq_motions_free_device)(
            lq, r, bufA.as<double>(), bufB.as<double>(), n, ns, o, ss, bufO.as<uint8_t>(),
            reinterpret_cast<unsigned long long *>(c.d_scalar + 5)))
        return rc;
    MPB_CUDA(cudaMemcpyAsync(out, bufO.p, (size_t)n, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaMemcpyAsync(c.h_scalar + 5, c.d_scalar + 5, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    if (checks) *checks = c.h_scalar[5];
    return MPB200_OK;
}

int mpb200_close_points(const mpb200_obstacles *o, const double *p_aos, const double *W, int64_t n, int dw, double r2,
                        int32_t *count, double *d2, int32_t *shape, double *x, double *all_d2, double *all_x) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(o != nullptr, "obstacle handle is NULL");
    MPB_CHECK_ARG(n >= 0 && dw >= 1, "bad batch size / dimension");
    MPB_CHECK_ARG(n == 0 || (p_aos && W && count && d2 && shape && x), "NULL buffers");
    const int64_t S = o->kind == 0 ? o->n_shapes : o->M;
    if (n == 0) return MPB200_OK;
    if (S == 0) { memset(count, 0, sizeof(int32_t) * (size_t)n); return MPB200_OK; }
    cudaStream_t st = ctx().stream;
    static DevBuf bP, bW, bC, bD, bS, bX, bAD, bAX;  // reused staging (single caller thread)
    const size_t nS = (size_t)(n * S);
    if (int rc = bP.reserve(sizeof(double) * (size_t)(n * dw))) return rc;
    if (int rc = bW.reserve(sizeof(double) * (size_t)(n * dw * dw))) return rc;
    if (int rc = bC.reserve(sizeof(int) * (size_t)n)) return rc;
    if (int rc = bD.reserve(sizeof(double) * nS)) return rc;
    if (int rc = bS.reserve(sizeof(int) * nS)) return rc;
    if (int rc = bX.reserve(sizeof(double) * nS * dw)) return rc;
    if (int rc = bAD.reserve(sizeof(double) * nS)) return rc;
    if (int rc = bAX.reserve(sizeof(double) * nS * dw)) return rc;
    MPB_CUDA(cudaMemcpyAsync(bP.p, p_aos, sizeof(double) * (size_t)(n * dw), cudaMemcpyHostToDevice, st));
    MPB_CUDA(cudaMemcpyAsync(bW.p, W, sizeof(double) * (size_t)(n * dw * dw), cudaMemcpyHostToDevice, st));
    MPB_CUDA(cudaMemsetAsync(bD.p, 0, sizeof(double) * nS, st));
    MPB_CUDA(cudaMemsetAsync(bS.p, 0xff, sizeof(int) * nS, st));
    MPB_CUDA(cudaMemsetAsync(bX.p, 0, sizeof(double) * nS * dw, st));
    if (int rc = close_points_device(o, bP.as<double>(), bW.as<double>(), n, dw, r2, bC.as<int>(), bD.as<double>(),
                                     bS.as<int>(), bX.as<double>(), bAD.as<double>(), bAX.as<double>()))
        return rc;
    MPB_CUDA(cudaMemcpyAsync(count, bC.p, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaMemcpyAsync(d2, bD.p, sizeof(double) * nS, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaMemcpyAsync(shape, bS.p, sizeof(int) * nS, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaMemcpyAsync(x, bX.p, sizeof(double) * nS * dw, cudaMemcpyDeviceToHost, st));
    if (all_d2) MPB_CUDA(cudaMemcpyAsync(all_d2, bAD.p, sizeof(double) * nS, cudaMemcpyDeviceToHost, st));
    if (all_x) MPB_CUDA(cudaMemcpyAsync(all_x, bAX.p, sizeof(double) * nS * dw, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    return MPB200_OK;
}

// ---- chopped-metric car spaces --------------------------------------------------------------------------------
int mpb200_car_inball_build(mpb200_samples *s, int32_t kind, double turning_radius, double r, double chopval,
                            mpb200_table **tableF, mpb200_table **tableB, int64_t *nnzF, int64_t *nnzB) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(s != nullptr && tableF != nullptr, "NULL handle");
    MPB_CHECK_ARG(s->d == 3, "car spaces need SE2 states (d = 3: x, y, theta)");
    MPB_CHECK_ARG(r >= 0 && r == r && chopval == chopval, "r must be a non-negative number");
    if (int rc = car_args(kind, turning_radius, 1.0)) return rc;
    MPB_CHECK_ARG(tableB == nullptr || (tableB != tableF && (*tableB == nullptr || *tableB != *tableF)),
                  "tableF and tableB must be different handles");
    // the (x, y) columns as a 2-D sample set (the reference's KD-tree lower-bound structure), made once
    if (!s->shadow_xy) {
        mpb200_samples *xy = new (std::nothrow) mpb200_samples();
        if (!xy) return fail(MPB200_ENOMEM, "out of host memory");
        xy->N = s->N; xy->d = 2; xy->q0 = 0; xy->q1 = s->N;
        int rc = xy->V.reserve(sizeof(double) * (size_t)(2 * s->N + 1));
        if (!rc) rc = car_extract_xy_device(s->V.as<double>(), s->N, xy->V.as<double>());
        if (!rc) rc = finish_samples(xy);
        if (rc) { mpb200_samples_destroy(xy); return rc; }
        s->shadow_xy = xy;
    }
    mpb200_samples *xy = s->shadow_xy;
    if (xy->q0 != s->q0 || xy->q1 != s->q1)
        if (int rc = mpb200_samples_set_query_range(xy, s->q0, s->q1)) return rc;
    if (int rc = mpb200_inball_build(xy, r, &s->shadow_cand, nullptr)) return rc;
    mpb200_table *tF = *tableF, *tB = tableB ? *tableB : nullptr;
    bool freshF = false, freshB = false;
    if (!tF) { tF = new (std::nothrow) mpb200_table(); freshF = true; }
    if (tableB && !tB) { tB = new (std::nothrow) mpb200_table(); freshB = true; }
    if (!tF || (tableB && !tB)) {
        if (freshF && tF) mpb200_table_destroy(tF);
        if (freshB && tB) mpb200_table_destroy(tB);
        return fail(MPB200_ENOMEM, "out of host memory");
    }
    int rc = car_inball_device(s, s->shadow_cand, kind, turning_radius, r, chopval, tF, tB, s->car_work, s->scan_tmp);
    if (rc) {
        if (freshF) mpb200_table_destroy(tF);
        if (freshB) mpb200_table_destroy(tB);
        return rc;
    }
    *tableF = tF;
    if (tableB) *tableB = tB;
    if (nnzF) *nnzF = tF->nnz;
    if (nnzB) *nnzB = tB ? tB->nnz : 0;
    return MPB200_OK;
}
int mpb200_car_last_candidates(const mpb200_samples *s, int64_t *pairs) {
    MPB_CHECK_ARG(s != nullptr && pairs != nullptr, "NULL argument");
    *pairs = s->shadow_cand ? s->shadow_cand->nnz : 0;
    return MPB200_OK;
}
int mpb200_car_steer(int32_t kind, double turning_radius, double speed, const double *v, const double *w, int64_t n,
                     double *cost, int32_t *nseg, double *segments) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(n >= 0 && (n == 0 || (v && w && cost && nseg && segments)), "NULL argument");
    if (int rc = car_args(kind, turning_radius, speed)) return rc;
    if (n == 0) return MPB200_OK;
    cudaStream_t st = ctx().stream;
    static DevBuf bufA, bufB, bufC, bufN, bufS;
    const size_t bytes = sizeof(double) * (size_t)(3 * n);
    if (int rc = bufA.reserve(bytes)) return rc;
    if (int rc = bufB.reserve(bytes)) return rc;
    if (int rc = bufC.reserve(sizeof(double) * (size_t)n)) return rc;
    if (int rc = bufN.reserve(sizeof(int) * (size_t)n)) return rc;
    if (int rc = bufS.reserve(sizeof(double) * (size_t)(15 * n))) return rc;
    MPB_CUDA(cudaMemcpyAsync(bufA.p, v, bytes, cudaMemcpyHostToDevice, st));
    MPB_CUDA(cudaMemcpyAsync(bufB.p, w, bytes, cudaMemcpyHostToDevice, st));
    if (int rc = car_steer_device(kind, turning_radius, speed, bufA.as<double>(), bufB.as<double>(), n, bufC.as<double>(),
                                  bufN.as<int>(), bufS.as<double>()))
        return rc;
    MPB_CUDA(cudaMemcpyAsync(cost, bufC.p, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaMemcpyAsync(nseg, bufN.p, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaMemcpyAsync(segments, bufS.p, sizeof(double) * (size_t)(15 * n), cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    return MPB200_OK;
}
int mpb200_car_edges_free(const mpb200_samples *s, const mpb200_table *t_, int32_t kind, double turning_radius,
                          double speed, const mpb200_obstacles *o, const mpb200_space_desc *ss, uint64_t *bitchunks,
                          int64_t *checks) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(s && t_ && o && ss, "NULL handle");
    MPB_CHECK_ARG(s->d == 3, "car spaces need SE2 states (d = 3: x, y, theta)");
    if (int rc = car_args(kind, turning_radius, speed)) return rc;
    mpb200_table *t = const_cast<mpb200_table *>(t_);
    MPB_CHECK_ARG(t->src_N == s->N && t->src_d == s->d, "the table was not built from this sample set");
    Context &c = ctx();
    cudaStream_t st = c.stream;
    const size_t words = (size_t)ceil_div(t->nnz, 64);
    if (int rc = t->edge_bits.reserve(sizeof(uint64_t) * (words + 1))) return rc;
    t->edge_bits_valid = false;
    phase_bank(MPB200_OP_EDGES);
    phase_mark(0);
    MPB_CUDA(cudaMemsetAsync(t->edge_bits.p, 0, sizeof(uint64_t) * (words + 1), st));
    MPB_CUDA(cudaMemsetAsync(c.d_scalar + 4, 0, sizeof(int64_t), st));
    if (int rc = car_edges_free_device(s, t, kind, turning_radius, speed, o, ss, t->edge_bits.as<uint32_t>(),
                                       reinterpret_cast<unsigned long long *>(c.d_scalar + 4)))
        return rc;
    t->edge_bits_valid = true;
    t->edge_bits_nnz = t->nnz;
    phase_mark(1);
    phases_collect(1);
    if (bitchunks || checks) {
        if (bitchunks && words)
            MPB_CUDA(cudaMemcpyAsync(bitchunks, t->edge_bits.p, sizeof(uint64_t) * words, cudaMemcpyDeviceToHost, st));
        MPB_CUDA(cudaMemcpyAsync(c.h_scalar + 4, c.d_scalar + 4, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        MPB_CUDA(cudaStreamSynchronize(st));
        if (checks) *checks = c.h_scalar[4];
    }
    return MPB200_OK;
}
int mpb200_car_motions_free(int32_t kind, double turning_radius, double speed, const double *v, const double *w,
                            int64_t n, const mpb200_obstacles *o, const mpb200_space_desc *ss, uint8_t *out,
                            int64_t *checks) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(o && ss && n >= 0 && (n == 0 || (v && w && out)), "NULL argument");
    if (int rc = car_args(kind, turning_radius, speed)) return rc;
    if (checks) *checks = 0;
    if (n == 0) return MPB200_OK;
    Context &c = ctx();
    cudaStream_t st = c.stream;
    static DevBuf bufA, bufB, bufO;
    const size_t bytes = sizeof(double) * (size_t)(3 * n);
    if (int rc = bufA.reserve(bytes)) return rc;
    if (int rc = bufB.reserve(bytes)) return rc;
    if (int rc = bufO.reserve((size_t)n + 64)) return rc;
    MPB_CUDA(cudaMemcpyAsync(bufA.p, v, bytes, cudaMemcpyHostToDevice, st));
    MPB_CUDA(cudaMemcpyAsync(bufB.p, w, bytes, cudaMemcpyHostToDevice, st));
    MPB_CUDA(cudaMemsetAsync(c.d_scalar + 5, 0, sizeof(int64_t), st));
    if (int rc = car_motions_free_device(kind, turning_radius, speed, bufA.as<double>(), bufB.as<double>(), n, o, ss,
                                         bufO.as<uint8_t>(), reinterpret_cast<unsigned long long *>(c.d_scalar + 5)))
        return rc;
    MPB_CUDA(cudaMemcpyAsync(out, bufO.p, (size_t)n, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaMemcpyAsync(c.h_scalar + 5, c.d_scalar + 5, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    if (checks) *checks = c.h_scalar[5];
    return MPB200_OK;
}

// ---- k-nearest connections (table operations) ----------------------------------------------------------------
static int out_table(mpb200_table **out, mpb200_table **t, bool *fresh) {
    *t = *out;
    *fresh = false;
    if (!*t) {
        *t = new (std::nothrow) mpb200_table();
        if (!*t) return fail(MPB200_ENOMEM, "out of host memory");
        *fresh = true;
    }
    return 0;
}
int mpb200_table_knn(const mpb200_table *t, int k, mpb200_table **out, int64_t *nnz, int64_t *short_cols) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(t != nullptr && out != nullptr, "NULL handle");
    MPB_CHECK_ARG(k >= 1, "k must be at least 1");
    MPB_CHECK_ARG(*out != t, "the output table must be a different handle");
    mpb200_table *o;
    bool fresh;
    if (int rc = out_table(out, &o, &fresh)) return rc;
    static DevBuf scan_tmp;
    int64_t n_short = 0;
    int rc = table_knn_device(t, k, o, &n_short, scan_tmp);
    if (rc) { if (fresh) mpb200_table_destroy(o); return rc; }
    *out = o;
    if (nnz) *nnz = o->nnz;
    if (short_cols) *short_cols = n_short;
    return MPB200_OK;
}
int mpb200_table_short_columns(const mpb200_table *t, int k, int64_t *short_cols) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(t != nullptr && short_cols != nullptr, "NULL argument");
    MPB_CHECK_ARG(k >= 1, "k must be at least 1");
    return table_short_columns_device(t, k, short_cols);
}
int mpb200_table_union_transpose(const mpb200_table *a, const mpb200_table *b, mpb200_table **out, int64_t *nnz) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(a != nullptr && b != nullptr && out != nullptr, "NULL handle");
    MPB_CHECK_ARG(*out != a && *out != b, "the output table must be a different handle");
    MPB_CHECK_ARG(a->src_N == b->src_N && a->src_N >= 0, "the two tables were built from different sample sets");
    MPB_CHECK_ARG(a->col0 == 0 && b->col0 == 0 && a->ncols == a->src_N && b->ncols == b->src_N,
                  "mutual neighbourhoods need full-range tables (every column of the sample set)");
    mpb200_table *o;
    bool fresh;
    if (int rc = out_table(out, &o, &fresh)) return rc;
    static DevBuf scan_tmp;
    int rc = table_union_transpose_device(a, b, o, scan_tmp);
    if (rc) { if (fresh) mpb200_table_destroy(o); return rc; }
    *out = o;
    if (nnz) *nnz = o->nnz;
    return MPB200_OK;
}

int mpb200_table_write_floor(const mpb200_table *t, double *ms) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(t != nullptr && ms != nullptr, "NULL argument");
    MPB_CHECK_ARG(t->ncols > 0 && t->nnz > 0, "empty table");
    return table_write_floor_device(t, ms);
}

int mpb200_pipe_peak(int kind, double *ops_per_s) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(ops_per_s != nullptr, "ops_per_s is NULL");
    MPB_CHECK_ARG(kind >= MPB200_PEAK_DADD_DMUL && kind <= MPB200_PEAK_FFMA, "unknown peak kind");
    return pipe_peak_device(kind, ops_per_s);
}

// ---- Monte-Carlo collision probability ---------------------------------------------------------
int mpb200_mc_collision_probability(const mpb200_mc_problem *p, const mpb200_obstacles *o, uint64_t seed, int64_t first,
                                    int64_t n, mpb200_mc_result *out, uint8_t *hit_out, double *w_out) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(p && o && out, "NULL argument");
    MPB_CHECK_ARG(p->T >= 1 && p->nz >= 1 && p->q >= 1 && p->dw >= 1 && p->K >= 0, "bad problem dimensions");
    MPB_CHECK_ARG(p->F && p->G && p->Wz && p->wbar && p->alpha && (p->K == 0 || p->mu), "NULL problem arrays");
    MPB_CHECK_ARG(n >= 0 && first >= 0, "negative rollout range");
    double sum = 0;
    for (int k = 0; k <= p->K; ++k) {
        MPB_CHECK_ARG(p->alpha[k] >= 0, "mixture weights must be non-negative");
        sum += p->alpha[k];
    }
    MPB_CHECK_ARG(sum > 0.999999 && sum < 1.000001 && p->alpha[0] > 0, "mixture weights must sum to 1 with alpha[0] > 0");
    double r4[4] = {0, 0, 0, 0};
    if (n > 0)
        if (int rc = mc_run_device(p, o, seed, first, n, r4, hit_out, w_out)) return rc;
    out->s1 = r4[0]; out->s2 = r4[1]; out->s0 = r4[2]; out->n = n; out->hits = (int64_t)(r4[3] + 0.5);
    return MPB200_OK;
}

}  // extern "C"
