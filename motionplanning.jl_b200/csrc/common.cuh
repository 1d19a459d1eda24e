// common.cuh -- runtime plumbing shared by every translation unit of libmpb200.so.
// Error convention, the per-process context (device, stream, timing events), device
// buffers that grow and are reused, and launch accounting.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdarg>
#include <cstring>
#include "../../include/mpb200.h"

namespace mpb {

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs
constexpr int kMaxPhases = 8;
constexpr int kBanks = 6;  // separate phase-event banks: MPB200_OP_TABLE / _POINTS / _EDGES / _OTHER / _PLAN / _PATH

struct Context {
    bool ready = false;
    int device = -1;
    int sm_count = kNumSMs;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;  // the launching stream (own or caller's)
    cudaEvent_t ev[kBanks][kMaxPhases + 1] = {};
    double last_ms[kBanks][kMaxPhases] = {};
    int pending_marks[kBanks] = {};  // phase events recorded but not yet turned into last_ms (done lazily: no sync in the call)
    int bank = 0;                    // bank of the operation in progress / most recent
    int64_t launches = 0;
    int64_t *d_scalar = nullptr;  // small device scratch for scalars read back to the host
    int64_t *h_scalar = nullptr;  // pinned mirror
    cudaEvent_t ev_scalar = nullptr;  // marks the end of a scalar read-back (waited on instead of the whole stream)
};
Context &ctx();

void set_error(const char *fmt, ...);
int fail(int code, const char *fmt, ...);

#define MPB_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess)                                                                 \
            return mpb::fail(MPB200_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                             __FILE__, __LINE__);                                               \
    } while (0)

#define MPB_REQUIRE_INIT()                                                             \
    do {                                                                               \
        if (!mpb::ctx().ready)                                                         \
            return mpb::fail(MPB200_ESTATE, "mpb200_init has not been called (no CPU fallback exists)"); \
    } while (0)

#define MPB_CHECK_ARG(cond, msg)                         \
    do {                                                 \
        if (!(cond)) return mpb::fail(MPB200_EARG, msg); \
    } while (0)

// count + check a kernel launch
#define MPB_LAUNCHED()                                                                            \
    do {                                                                                          \
        mpb::ctx().launches++;                                                                    \
        mpb::trace_mark(__FILE__, __LINE__);                                                      \
        cudaError_t e__ = cudaGetLastError();                                                     \
        if (e__ != cudaSuccess)                                                                   \
            return mpb::fail(MPB200_ECUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), \
                             __FILE__, __LINE__);                                                 \
    } while (0)

// A device buffer that only grows; reused across calls so the steady state has no cudaMalloc.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes);
    void release();
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

size_t cache_parked_bytes();  // device bytes parked in the block cache (free for the next reserve)
uint64_t next_serial();       // process-unique id of a new sample set

// timing phases: phase_begin(0) ... phase_end(0) record events on the launching stream
void phase_bank(int op);               // select the event bank of the operation that starts now
int phase_mark(int i);                 // record event i
// MPB200_TRACE=1: an event after every kernel launch (no graph), per-launch gaps printed by trace_dump()
void trace_mark(const char *file, int line);
void trace_dump();
int phases_collect(int n_marks);       // note n_marks events; mpb200_last_ms() waits for them and computes last_ms

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

}  // namespace mpb

// ---- handle layouts (opaque in the C ABI) ---------------------------------------
struct mpb200_xchg;
struct mpb200_table;
namespace mpb {
// xchg.cu: start sending an attached table's column lengths right after its count scan (side stream)
int xchg_push_counts_early(mpb200_xchg *x, const mpb200_table *t, const int64_t *colptr, int64_t ncols);
}
struct mpb200_table {
    mpb200_xchg *xchg = nullptr;  // exchange this table's builds feed (mpb200_xchg_attach), or NULL
    int64_t ncols = 0;     // columns in this shard
    int64_t col0 = 0;      // first global column (0-based)
    int64_t nnz = 0;
    double r = 0;
    bool euclid = false;   // Euclidean r-ball table: every stored neighbour lies within r of its column point
    mpb::DevBuf colptr;    // int64 (ncols+1), 1-based, relative to the shard
    mpb::DevBuf rowval;    // int64 nnz, 1-based global row ids
    mpb::DevBuf nzval;     // f64 nnz
    mpb::DevBuf counts;    // int32 ncols (scratch)
    mpb::DevBuf masks;     // per-query hit lists (one byte per hit, 64 B/query; scratch between count and fill)
    mpb::DevBuf edge_bits; // uint64 ceil(nnz/64): last mpb200_edges_free result
    mpb::DevBuf scratch;   // big-column spill etc.
    mpb::DevBuf col_list;  // int32 ncols: columns classify_columns leaves for the per-edge test (scratch)
    mpb::DevBuf col_order; // int32 ncols: the shard's columns in grid-cell order (spatially coherent warps)
    bool has_order = false;
    uint64_t grid_build = 0;  // the samples' grid build that made col_order (its cell-ordered copy matches while equal)
    bool edge_bits_valid = false;  // edge_bits describes the CURRENT table contents (cleared by every build)
    int64_t edge_bits_nnz = 0;
    int64_t src_N = -1;            // the sample set the table was built from (rowval addresses its samples)
    int src_d = 0;
    uint64_t src_serial = 0;       // ... and its serial
};

struct mpb200_samples {
    uint64_t serial = mpb::next_serial();  // tells tables built from this set from those built from another of equal size
    int64_t N = 0;
    int d = 0;
    int64_t q0 = 0, q1 = 0;
    mpb::DevBuf V;           // f64 d x N column-major (AoS), as the caller gave it
    // uniform grid (built per radius by mpb200_inball_build)
    mpb::DevBuf cell_start;  // int32 ncells+1
    mpb::DevBuf cell_fill;   // int32 ncells+1: per-cell histogram (its atomics hand out the in-cell ranks)
    mpb::DevBuf sorted_idx;  // int32 N   original index of the k-th point in cell order
    mpb::DevBuf sorted_pos;  // f64 d x N positions in cell order (AoS)
    mpb::DevBuf pt_order;    // int32 (q1-q0): the shard's samples (relative to q0) in grid-cell order, from the last grid build
    bool pt_order_valid = false;  // sorted_pos, sorted_idx, q_order and pt_order still hold the last grid build
    uint64_t grid_build = 0;      // serial of the last grid build
    bool sorted_x = false;   // samples are non-decreasing along the first coordinate (checked once at create)
    mpb::DevBuf minmax;      // f64 2*d bounding box
    double h_bbox[32] = {};  // host copy of the bounding box (mins then maxs), read once at create
    double h_qbbox[32] = {}; // bounding box of the query range's samples (== h_bbox for the full range)
    mpb::DevBuf scan_tmp;    // scan block sums
    mpb::DevBuf q_order;     // int32: cell-order positions owned by this shard (+ scratch)
    mpb::DevBuf point_bits;  // uint64 ceil(N/64): last mpb200_points_free result
    bool point_bits_valid = false;  // point_bits hold the validity of all N samples (the last call covered [0, N))
    mpb::DevBuf aux;         // small per-build constants (e.g. the centring vector of the tensor-core path)
    // CUDA graph of the launch-bound front half of a grid build (K1 + count + scans), replayed
    // while the launch parameters (sizes, radius, buffer addresses) stay the same
    cudaGraphExec_t graph_exec = nullptr;
    uint64_t graph_key[32] = {};
    int graph_launches = 0;  // kernels inside the graph (launch accounting)
    // car spaces (cars.cu): the (x, y) columns as a sample set of their own + the Euclidean candidate table over them
    mpb200_samples *shadow_xy = nullptr;
    mpb200_table *shadow_cand = nullptr;
    mpb::DevBuf car_work;
};

struct mpb200_obstacles {
    int kind = 0;            // 0 = 2-D compound, 1 = N-d boxes
    // 2-D compound, packed for the device: see predicates.cuh
    int n_gates = 0, n_shapes = 0, flags = 0;
    int table_words = 0;     // size of the packed table in doubles
    mpb::DevBuf table;       // packed f64 table
    // boxes
    int M = 0, d = 0;
};

namespace mpb {
constexpr int kLqgMaxN = 6;  // state / control dimension limit of the general linear-affine path
// per-system tables of the general path (lq_general.cu; same content as the oracle's orc_lqg), row-major
struct LqgHost {
    int n = 0, np = 0;
    double A[kLqgMaxN * kLqgMaxN], c[kLqgMaxN], BRB[kLqgMaxN * kLqgMaxN];
    double Ak[kLqgMaxN][kLqgMaxN * kLqgMaxN], dk[kLqgMaxN][kLqgMaxN];
    double Gp[2 * kLqgMaxN][kLqgMaxN * kLqgMaxN];
};
}  // namespace mpb

struct mpb200_lq {
    int d = 0;              // double-integrator closed form (lq.cu): position dimension; state dimension n = 2 d
    bool scalar_R = false;  // R == rho * I
    double R[9] = {};       // d x d row-major (symmetric)
    bool general = false;   // any other nilpotent (A, B, c): numeric 2BVP of lq_general.cu
    mpb::LqgHost gen;       // its tables on the host ...
    mpb::DevBuf gen_dev;    // ... and on the device (layout LqgTab<n>)
};
