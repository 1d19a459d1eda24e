// collide.cu -- K6 (batched point validity), K7 (batched segment vs 2-D compound) and
// K8 (batched segment vs N-d box list).
//
// Replaces the per-call loops of the reference: F[i] = is_free_state(V[i], CC, SS)
// (fmt.jl:31-36, sampling.jl:25) and the lazy is_free_motion(V[y], V[x], CC, SS) of fmt.jl:75,
// batched over every stored entry of a neighbour table.  One lane per point / edge, the
// obstacle table staged once per CTA into shared memory, results packed into Julia BitVector words
// (bit k&63 of word k>>6 == bit k&31 of 32-bit word k>>5, little endian).  After a grid build the
// points and the columns are visited in grid-cell order, read from the build's cell-ordered copy of
// the samples (the lanes of a warp then agree on which obstacles they are near); classify_columns
// settles whole columns whose r-box is clear of every obstacle (or inside one convex polygon) and only
// the rest reach the per-edge kernel.
#include "common.cuh"
#include "predicates.cuh"
#include "philox.cuh"
#include "scan.cuh"
#include "gmt.cuh"
#include "shortcut.cuh"
#include <climits>
#include <cstdlib>

namespace mpb {

constexpr int kThreads = 256;

__device__ __forceinline__ const double *stage_table(const double *__restrict__ g_table, int words, bool use_smem,
                                                     double *smem) {
    if (!use_smem) return g_table;
    for (int i = threadIdx.x; i < words; i += blockDim.x) smem[i] = g_table[i];
    __syncthreads();
    return smem;
}

// is_free_state(v, CC, SS): statespaces.jl:151-152
template <int N, int DW, int KIND>
__device__ __forceinline__ bool state_free(const SpaceDev &S, const double *T, int M, const double *v) {
    if (!in_state_space<N>(S, v)) return false;
    double p[DW];
    state2workspace<N, DW>(S, v, p);
    if (KIND == 0) return !point_colliding_2d(T, p[0], p[DW > 1 ? 1 : 0]);
    return box_point_free<DW>(T, M, p);
}
// is_free_motion(v, w, CC, SS) with waypoints (v, w): statespaces.jl:153-158, geometric.jl:20.
// `checked` reports whether the segment test ran (CC.count += 1, robots2D.jl:13 / boxesND.jl:26).
template <int N, int DW, int KIND>
__device__ __forceinline__ bool motion_free(const SpaceDev &S, const double *T, int M, const double *v,
                                            const double *w, bool *checked) {
    *checked = false;
    if (!in_state_space<N>(S, v)) return false;  // the last waypoint is never bounds-checked (Q4)
    double p[DW], q[DW];
    state2workspace<N, DW>(S, v, p);
    state2workspace<N, DW>(S, w, q);
    *checked = true;
    if (KIND == 0) return !line_colliding_2d(T, p[0], p[DW > 1 ? 1 : 0], q[0], q[DW > 1 ? 1 : 0]);
    return box_segment_free<DW>(T, M, p, q);
}

// The grid build's cell-ordered copy of the sample set (grid_rball.cu): position t of the shard's cell-order
// walk holds sample q0 + pt_order[t] at sorted_pos[pos], pos = q_order ? q_order[t] : t.
struct CellOrder {
    const double *pos;    // sorted_pos (N x d, AoS)
    const int *q_order;   // shard: cell-order positions owned by the shard; NULL for the full range
    const int *pt_order;  // sample (relative to q0) at walk position t
};

template <int N, int DW, int KIND>
__global__ void __launch_bounds__(kThreads)
points_free_kernel(const double *__restrict__ V, int64_t n, SpaceDev S, const double *__restrict__ g_table,
                   int table_words, int M, bool use_smem, uint32_t *__restrict__ bits32,
                   uint8_t *__restrict__ bytes, CellOrder co) {
    extern __shared__ double s_table[];
    const double *T = stage_table(g_table, table_words, use_smem, s_table);
    const int64_t n_pad = (n + 31) & ~int64_t(31);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    if (N <= 3 && co.pos) {  // grid builds cover d = 2, 3
        // points visited in grid-cell order, read from the cell-ordered copy (coalesced): a warp's points are
        // neighbours, so its lanes agree on which obstacles they are near; bits land in the pre-zeroed words with
        // atomicOr.  The next point's loads are issued before the current point is tested.
        int64_t ti = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        double v[N];
        int64_t i = 0;
        if (ti < n) {
            const int64_t pos = co.q_order ? co.q_order[ti] : ti;
#pragma unroll
            for (int k = 0; k < N; ++k) v[k] = co.pos[pos * N + k];
            i = co.pt_order[ti];
        }
        while (ti < n) {
            const int64_t tn = ti + stride;
            double vn[N];
            int64_t in = 0;
            if (tn < n) {
                const int64_t pos = co.q_order ? co.q_order[tn] : tn;
#pragma unroll
                for (int k = 0; k < N; ++k) vn[k] = co.pos[pos * N + k];
                in = co.pt_order[tn];
            }
            const bool ok = state_free<N, DW, KIND>(S, T, M, v);
            if (bits32 && ok) atomicOr(&bits32[i >> 5], 1u << (i & 31));
            if (bytes) bytes[i] = ok ? 1 : 0;
            ti = tn; i = in;
#pragma unroll
            for (int k = 0; k < N; ++k) v[k] = vn[k];
        }
        return;
    }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pad; i += (int64_t)gridDim.x * blockDim.x) {
        bool ok = false;
        if (i < n) {
            double v[N];
#pragma unroll
            for (int k = 0; k < N; ++k) v[k] = V[i * N + k];
            ok = state_free<N, DW, KIND>(S, T, M, v);
        }
        unsigned m = __ballot_sync(0xffffffffu, ok);
        if (bits32 && (threadIdx.x & 31) == 0) bits32[i >> 5] = m;
        if (bytes && i < n) bytes[i] = ok ? 1 : 0;
    }
}

// The 2-D compound's cull boxes for warp_line_colliding_2d: lane s keeps box s in registers (S <= 32).
struct LaneCull {
    double xl, xh, yl, yh;
};
template <int KIND>
__device__ __forceinline__ LaneCull lane_cull(const Obs2 &O) {
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    LaneCull c{inf, -inf, inf, -inf};
    const int lane = threadIdx.x & 31;
    if (KIND == 0 && lane < O.S && O.S <= 32) {
        const double *cb = O.cull_box(lane);
        c = LaneCull{cb[0], cb[1], cb[2], cb[3]};
    }
    return c;
}

// Per-edge test of the stored entries [beg, end) of one column (row y -> column x), i.e. edges sharing the
// endpoint x whose workspace image is q: the 32 lanes take 32 entries at a time (coherent control flow, no
// per-edge search for the column).  y0 is rowval[beg + lane] - 1 where beg + lane < end, loaded by the caller
// ahead of time.  Validity bits go to the (pre-zeroed) BitVector words with at most two atomicOr per 32 edges.
template <int N, int DW, int KIND>
__device__ __forceinline__ void column_edges(const SpaceDev &S, const double *T, int M, const Obs2 &O,
                                             const LaneCull &cl, const double *__restrict__ V,
                                             const int64_t *__restrict__ rowval, int64_t beg, int64_t end,
                                             const double *q, int64_t y0, uint32_t *__restrict__ bits32,
                                             unsigned long long &my_checks) {
    const int lane = threadIdx.x & 31;
    for (int64_t e0 = beg; e0 < end; e0 += 32) {
        const int64_t e = e0 + lane;
        bool run = false;
        double a[N], p[DW];
#pragma unroll
        for (int k = 0; k < N; ++k) a[k] = 0.0;
        if (e < end) {
            const int64_t y = e0 == beg ? y0 : rowval[e] - 1;
#pragma unroll
            for (int k = 0; k < N; ++k) a[k] = V[y * N + k];
            run = in_state_space<N>(S, a);  // statespaces.jl:155: in_state_space(wps[1]) && segment test
        }
        state2workspace<N, DW>(S, a, p);
        my_checks += run ? 1 : 0;
        // warp-collective: every lane must make the call (no short-circuit on `run`)
        bool seg_free;
        if (KIND == 0)
            seg_free = !warp_line_colliding_2d(O, cl.xl, cl.xh, cl.yl, cl.yh, p[0], p[DW > 1 ? 1 : 0], q[0],
                                               q[DW > 1 ? 1 : 0], run);
        else
            seg_free = warp_box_segment_free<DW>(T, M, p, q, run);
        const bool ok = run && seg_free;
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        if (lane == 0 && m) {
            const int sh = (int)(e0 & 31);
            const int64_t wi = e0 >> 5;
            atomicOr(&bits32[wi], m << sh);
            if (sh && (m >> (32 - sh))) atomicOr(&bits32[wi + 1], m >> (32 - sh));
        }
    }
}

// per-CTA reduction of the CC.count increment, then one atomicAdd
__device__ __forceinline__ void add_checks(unsigned long long my_checks, unsigned long long *checks) {
    __shared__ unsigned long long s_checks[kThreads / 32];
#pragma unroll
    for (int o = 16; o; o >>= 1) my_checks += __shfl_xor_sync(0xffffffffu, my_checks, o);
    if ((threadIdx.x & 31) == 0) s_checks[threadIdx.x >> 5] = my_checks;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < kThreads / 32; ++w) t += s_checks[w];
        if (t) atomicAdd(checks, t);
    }
}

// One warp per column of the table (any table, any state-to-workspace map), in column order -- or, after
// classify_columns, per column of its list (length on the device).  The next column's colptr pair is prefetched while
// the current one is processed.
template <int N, int DW, int KIND>
__global__ void __launch_bounds__(kThreads, (DW <= 3) ? 3 : 1)
edges_free_kernel(const double *__restrict__ V, const int64_t *__restrict__ colptr,
                  const int64_t *__restrict__ rowval, int64_t ncols, int64_t col0, SpaceDev S,
                  const double *__restrict__ g_table, int table_words, int M, bool use_smem,
                  uint32_t *__restrict__ bits32, unsigned long long *__restrict__ checks,
                  const int *__restrict__ col_list, const unsigned long long *__restrict__ n_list) {
    extern __shared__ double s_table[];
    const double *T = stage_table(g_table, table_words, use_smem, s_table);
    const int lane = threadIdx.x & 31;
    const int64_t n_items = col_list ? (int64_t)*n_list : ncols;
    const int64_t gwarp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    unsigned long long my_checks = 0;
    Obs2 O(KIND == 0 ? T : nullptr, KIND == 0);
    const LaneCull cl = lane_cull<KIND>(O);
    int64_t it = gwarp, c = 0, beg = 0, end = 0;
    if (it < n_items) { c = col_list ? col_list[it] : it; beg = colptr[c] - 1; end = colptr[c + 1] - 1; }
    while (it < n_items) {
        const int64_t itn = it + nwarps;
        int64_t cn = 0, begn = 0, endn = 0;
        if (itn < n_items) { cn = col_list ? col_list[itn] : itn; begn = colptr[cn] - 1; endn = colptr[cn + 1] - 1; }  // prefetch
        if (beg < end) {
            const int64_t y0 = beg + lane < end ? rowval[beg + lane] - 1 : 0;
            double b[N], q[DW];
#pragma unroll
            for (int k = 0; k < N; ++k) b[k] = V[(col0 + c) * N + k];
            state2workspace<N, DW>(S, b, q);  // the last waypoint is never bounds-checked (Q4)
            column_edges<N, DW, KIND>(S, T, M, O, cl, V, rowval, beg, end, q, y0, bits32, my_checks);
        }
        it = itn; c = cn; beg = begn; end = endn;
    }
    add_checks(my_checks, checks);
}

// Column classes of a Euclidean r-ball table (state == workspace): every stored neighbour lies within r of the
// column point x, so all edges of the column live inside the box x +- r.
enum : int { kColFree = 0, kColColliding = 1, kColEdges = 2 };
// If the box is inside the state bounds and overlaps no obstacle's cull box, every edge passes in_state_space
// and is rejected by every obstacle's own AABB gate: the whole column is free.  If (2-D) the box sits inside one
// convex polygon, every edge collides.  Anything else needs the per-edge test.
template <int DW, int KIND>
__device__ __forceinline__ int classify_column(const SpaceDev &S, const double *T, int M, double r, const double *x) {
    double lo[DW], hi[DW];
    bool trivial = true;
#pragma unroll
    for (int i = 0; i < DW; ++i) {
        const double pad = r * (1.0 + 1e-9) + 4.5e-16 * fabs(x[i]);  // covers every rounding in x +- r
        lo[i] = x[i] - pad; hi[i] = x[i] + pad;
        trivial = trivial && (S.lo[i] <= lo[i] && hi[i] <= S.hi[i]);
    }
    if (!trivial) return kColEdges;
    if (KIND == 0) {
        Obs2 O(T);
        const double ylo = lo[DW > 1 ? 1 : 0], yhi = hi[DW > 1 ? 1 : 0];
        for (int s = 0; s < O.S; ++s) {
            const double *cb = O.cull_box(s);
            if (!(overlapping(lo[0], hi[0], cb[0], cb[1]) && overlapping(ylo, yhi, cb[2], cb[3]))) continue;
            trivial = false;
            // Both endpoints of every edge of the column lie in the box; if the box is inside
            // polygon s by a margin far above rounding, no axis of the SAT test separates
            // (SAT2D.jl:172-176), so every edge collides -- given the gate chain passes, which
            // holds for consistent gates because they contain the polygon's AABB.
            if (O.kind(s) == 1 && O.consistent()) {
                const double *P = O.data(s);
                const int K = O.K(s);
                const double *nrm = P + 4 + 2 * K, *ext = P + 4 + 4 * K;
                const double m = 1e-9 * (1.0 + fabs(lo[0]) + fabs(hi[0]) + fabs(ylo) + fabs(yhi));
                bool inside = true;
                for (int i = 0; i < K && inside; ++i) {
                    const double n1 = nrm[2 * i], n2 = nrm[2 * i + 1];
                    const double dmax = fmax(lo[0] * n1, hi[0] * n1) + fmax(ylo * n2, yhi * n2);
                    inside = dmax <= ext[2 * i + 1] - m;  // support of the box along the outward normal
                }
                if (inside) return kColColliding;
            }
        }
        return trivial ? kColFree : kColEdges;
    }
    const double *bl = T, *bh = T + (size_t)M * DW;
    for (int k = 0; k < M; ++k) {
        bool sep = false;
#pragma unroll
        for (int i = 0; i < DW; ++i) sep = sep || (bh[k * DW + i] < lo[i] || bl[k * DW + i] > hi[i]);
        if (!sep) return kColEdges;
    }
    return kColFree;
}

// One lane per column of a Euclidean r-ball table with an identity state-to-workspace map, in grid-cell order when
// the table has one (the lanes of a warp then look at neighbouring points and take the same branches), from a grid
// of resident CTAs.  The column point comes from the grid build's cell-ordered copy when it describes this table
// (a coalesced read), else from V.  The next column's id, colptr pair and point are loaded before the current one
// is classified.  Free columns get their bits here (<= 3 atomicOr) and colliding ones nothing; both advance
// `checks` by the column length.  The rest are appended to `list` (one atomicAdd per warp) for edges_free_kernel.
// counters: [0] segment tests run (CC.count), [1] list length -- zeroed before the launch.
template <int DW, int KIND>
__global__ void __launch_bounds__(kThreads)
classify_columns(const double *__restrict__ V, const int64_t *__restrict__ colptr, int64_t ncols, int64_t col0,
                 double r, SpaceDev S, const double *__restrict__ g_table, int table_words, int M, bool use_smem,
                 const int *__restrict__ col_order, CellOrder co, uint32_t *__restrict__ bits32,
                 unsigned long long *__restrict__ counters, int *__restrict__ list) {
    extern __shared__ double s_table[];
    const double *T = stage_table(g_table, table_words, use_smem, s_table);
    const int lane = threadIdx.x & 31;
    unsigned long long my_checks = 0;
    unsigned long long *bits64 = reinterpret_cast<unsigned long long *>(bits32);
    const double *P = co.pos ? co.pos : V;
    const int64_t n_pad = (ncols + 31) & ~int64_t(31);  // whole warps: the ballot below needs every lane
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    // walk position t -> column c, its stored entries [beg, end) and its point
    auto load = [&](int64_t t, int64_t &c, int64_t &beg, int64_t &end, double *x) {
        beg = end = 0;
        if (t < ncols) {
            c = col_order ? col_order[t] : t;
            beg = colptr[c] - 1; end = colptr[c + 1] - 1;
            const int64_t xo = (co.pos ? (co.q_order ? co.q_order[t] : t) : col0 + c) * DW;
#pragma unroll
            for (int i = 0; i < DW; ++i) x[i] = P[xo + i];
        }
    };
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t c = 0, beg, end;
    double x[DW];
    load(t, c, beg, end, x);
    while (t < n_pad) {
        const int64_t tn = t + stride;
        int64_t cn = 0, begn, endn;
        double xn[DW];
        load(tn, cn, begn, endn, xn);  // prefetch
        const int cls = beg < end ? classify_column<DW, KIND>(S, T, M, r, x) : kColFree;
        if (cls != kColEdges) my_checks += (unsigned long long)(end - beg);  // colliding: every test runs and fails
        if (cls == kColFree) {
            for (int64_t w = beg >> 6; beg < end && w <= (end - 1) >> 6; ++w) {
                const int64_t b0 = w << 6;
                const int from = (int)(beg > b0 ? beg - b0 : 0), to = (int)(end < b0 + 64 ? end - b0 : 64);
                const unsigned long long m = (to - from == 64) ? ~0ULL : (((1ULL << (to - from)) - 1ULL) << from);
                atomicOr(&bits64[w], m);
            }
        }
        const unsigned fm = __ballot_sync(0xffffffffu, cls == kColEdges);
        if (fm) {
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(&counters[1], (unsigned long long)__popc(fm));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (cls == kColEdges) list[base + __popc(fm & ((1u << lane) - 1u))] = (int)c;
        }
        t = tn; c = cn; beg = begn; end = endn;
#pragma unroll
        for (int i = 0; i < DW; ++i) x[i] = xn[i];
    }
    add_checks(my_checks, &counters[0]);
}

template <int N, int DW, int KIND>
__global__ void __launch_bounds__(kThreads)
segments_free_kernel(const double *__restrict__ A, const double *__restrict__ B, int64_t n, SpaceDev S,
                     const double *__restrict__ g_table, int table_words, int M, bool use_smem,
                     uint8_t *__restrict__ out) {
    extern __shared__ double s_table[];
    const double *T = stage_table(g_table, table_words, use_smem, s_table);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double a[N], b[N];
#pragma unroll
        for (int k = 0; k < N; ++k) { a[k] = A[i * N + k]; b[k] = B[i * N + k]; }
        bool checked;
        out[i] = motion_free<N, DW, KIND>(S, T, M, a, b, &checked) ? 1 : 0;
    }
}

// ---- host dispatch --------------------------------------------------------------------
constexpr size_t kSmemTableMax = 160 * 1024;

// ---- batched free-state sampling (SURVEY 8(f).1; sample_free!, sampling.jl:23-37) ---------------------------
// Candidate c of the stream (oracle/sample.c): coordinate i = lo_i + u (hi_i - lo_i) with u the 53-bit uniform
// from Philox4x32-10(counter = (c lo, c hi, i / 2, 'SAMP'), key = seed); kept iff is_free_state.
template <int N>
__device__ __forceinline__ void sample_candidate(const SpaceDev &S, uint32_t k0, uint32_t k1, int64_t c, double *x) {
    const Philox ph{k0, k1};
#pragma unroll
    for (int b = 0; 2 * b < N; ++b) {
        uint32_t rnd[4];
        ph((uint32_t)c, (uint32_t)((uint64_t)c >> 32), (uint32_t)b, 0x53414D50u, rnd);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int i = 2 * b + h;
            if (i < N) x[i] = dadd(S.lo[i], dmul(u53(rnd[2 * h], rnd[2 * h + 1]), dsub(S.hi[i], S.lo[i])));
        }
    }
}
template <int N, int DW, int KIND>
__global__ void __launch_bounds__(kThreads)
sample_flags_kernel(SpaceDev S, const double *__restrict__ g_table, int table_words, int M, bool use_smem,
                    uint32_t k0, uint32_t k1, int64_t c0, int64_t C, int *__restrict__ flags) {
    extern __shared__ double s_table[];
    const double *T = stage_table(g_table, table_words, use_smem, s_table);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < C; i += (int64_t)gridDim.x * blockDim.x) {
        double x[N];
        sample_candidate<N>(S, k0, k1, c0 + i, x);
        flags[i] = state_free<N, DW, KIND>(S, T, M, x) ? 1 : 0;
    }
}
// free candidate i of the chunk becomes sample base + offs[i] (candidate order is kept); the candidate is regenerated
// instead of being stored; the thread that writes sample n_want - 1 reports how many candidates that took
template <int N>
__global__ void __launch_bounds__(kThreads)
sample_scatter_kernel(SpaceDev S, uint32_t k0, uint32_t k1, int64_t c0, int64_t C, const int *__restrict__ flags,
                      const int *__restrict__ offs, int64_t base, int64_t n_want, double *__restrict__ V,
                      long long *__restrict__ used) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < C; i += (int64_t)gridDim.x * blockDim.x) {
        if (!flags[i]) continue;
        const int64_t pos = base + offs[i];
        if (pos >= n_want) continue;
        double x[N];
        sample_candidate<N>(S, k0, k1, c0 + i, x);
#pragma unroll
        for (int k = 0; k < N; ++k) V[pos * N + k] = x[k];
        if (pos == n_want - 1) *used = c0 + i + 1;
    }
}

struct LaunchCfg {
    const double *table;
    int words, M;
    bool use_smem;
    size_t smem;
    unsigned grid;
};
static LaunchCfg make_cfg(const mpb200_obstacles *o, int64_t work) {
    LaunchCfg L;
    L.table = o->table.as<double>();
    L.words = o->table_words;
    L.M = o->M;
    size_t bytes = sizeof(double) * (size_t)o->table_words;
    L.use_smem = bytes <= kSmemTableMax;
    L.smem = L.use_smem ? bytes : 0;
    int64_t blocks = ceil_div(work > 0 ? work : 1, kThreads);
    int64_t cap = (int64_t)ctx().sm_count * 16;  // persistent-style grid: a multiple of the SM count
    L.grid = (unsigned)(blocks < cap ? blocks : cap);
    return L;
}
template <class K>
static int prep_kernel(K kernel, size_t smem) {
    if (smem > 48 * 1024) MPB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return 0;
}

// Grid of the validity kernels (K6, K7/K8): every thread loops over its items, so one wave of resident CTAs
// does the work -- as many as the occupancy calculator fits on the GPU at this shared-memory size, fewer when
// there are fewer than that many CTAs' worth of items.  Call after prep_kernel (it sets the shared-memory limit).
template <class K>
static int resident_grid(K kernel, size_t smem, int64_t items, unsigned *grid) {
    // the last answer per kernel signature, keyed by the kernel itself too: the instantiations of a template share one
    // signature (hence these statics) but not their register use; the occupancy query is a host call per launch otherwise
    static const void *cached_kernel = nullptr;
    static size_t cached_smem = ~size_t(0);
    static int per_sm = 0;
    if (smem != cached_smem || (const void *)kernel != cached_kernel) {
        MPB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, smem));
        if (per_sm < 1) per_sm = 1;
        cached_smem = smem;
        cached_kernel = (const void *)kernel;
    }
    const int64_t cap = (int64_t)per_sm * ctx().sm_count;
    const int64_t blocks = ceil_div(items > 0 ? items : 1, kThreads);
    *grid = (unsigned)(blocks < cap ? blocks : cap);
    return 0;
}

int make_space(const mpb200_space_desc *ss, int d_state, SpaceDev *out, int *dw) {
    MPB_CHECK_ARG(ss != nullptr, "space descriptor is NULL");
    MPB_CHECK_ARG(ss->n == d_state, "space dimension does not match the sample dimension");
    MPB_CHECK_ARG(ss->n >= 1 && ss->n <= kMaxDim, "state dimension out of range (1..16)");
    MPB_CHECK_ARG(ss->lo && ss->hi, "space bounds are NULL");
    SpaceDev S;
    memset(&S, 0, sizeof(S));
    S.n = ss->n;
    S.s2w_kind = ss->s2w_kind;
    for (int i = 0; i < ss->n; ++i) { S.lo[i] = ss->lo[i]; S.hi[i] = ss->hi[i]; }
    if (ss->s2w_kind == 0) {
        S.dw = ss->n;
    } else if (ss->s2w_kind == 1) {
        MPB_CHECK_ARG(ss->inds && ss->dw >= 1 && ss->dw <= kMaxDim, "VectorView needs inds and 1 <= dw <= 16");
        S.dw = ss->dw;
        for (int i = 0; i < ss->dw; ++i) {
            MPB_CHECK_ARG(ss->inds[i] >= 0 && ss->inds[i] < ss->n, "VectorView index out of range");
            S.inds[i] = ss->inds[i];
        }
    } else if (ss->s2w_kind == 2) {
        MPB_CHECK_ARG(ss->C && ss->dw >= 1 && ss->dw * ss->n <= kMaxDim * 4, "OutputMatrix needs C with dw*n <= 64");
        S.dw = ss->dw;
        for (int i = 0; i < ss->dw * ss->n; ++i) S.C[i] = ss->C[i];
    } else {
        return fail(MPB200_EARG, "unknown s2w_kind %d", ss->s2w_kind);
    }
    *out = S;
    *dw = S.dw;
    return 0;
}

// (N, DW) pairs compiled: Identity spaces N == DW in 2..10, and double-integrator style
// position views (4,2), (6,3).
#define MPB_DISPATCH_DIMS(N_, DW_, KIND_, CALL)                                            \
    do {                                                                                   \
        bool done__ = false;                                                               \
        if (KIND_ == 0) {                                                                  \
            if (DW_ != 2) return fail(MPB200_EARG, "2-D obstacles need a 2-D workspace");  \
            if (N_ == 2) { CALL(2, 2, 0); done__ = true; }                                 \
            else if (N_ == 3) { CALL(3, 2, 0); done__ = true; }                            \
            else if (N_ == 4) { CALL(4, 2, 0); done__ = true; }                            \
            else if (N_ == 6) { CALL(6, 2, 0); done__ = true; }                            \
        } else {                                                                           \
            if (N_ == 2 && DW_ == 2) { CALL(2, 2, 1); done__ = true; }                     \
            else if (N_ == 3 && DW_ == 3) { CALL(3, 3, 1); done__ = true; }                \
            else if (N_ == 4 && DW_ == 4) { CALL(4, 4, 1); done__ = true; }                \
            else if (N_ == 5 && DW_ == 5) { CALL(5, 5, 1); done__ = true; }                \
            else if (N_ == 6 && DW_ == 6) { CALL(6, 6, 1); done__ = true; }                \
            else if (N_ == 7 && DW_ == 7) { CALL(7, 7, 1); done__ = true; }                \
            else if (N_ == 8 && DW_ == 8) { CALL(8, 8, 1); done__ = true; }                \
            else if (N_ == 9 && DW_ == 9) { CALL(9, 9, 1); done__ = true; }                \
            else if (N_ == 10 && DW_ == 10) { CALL(10, 10, 1); done__ = true; }            \
            else if (N_ == 3 && DW_ == 2) { CALL(3, 2, 1); done__ = true; }                \
            else if (N_ == 4 && DW_ == 2) { CALL(4, 2, 1); done__ = true; }                \
            else if (N_ == 6 && DW_ == 3) { CALL(6, 3, 1); done__ = true; }                \
        }                                                                                  \
        if (!done__)                                                                       \
            return fail(MPB200_EARG, "unsupported (state dim %d, workspace dim %d) combination", N_, DW_); \
    } while (0)

static int check_obstacles(const mpb200_obstacles *o, int dw) {
    MPB_CHECK_ARG(o != nullptr, "obstacle handle is NULL");
    if (o->kind == 1 && o->d != dw) return fail(MPB200_EARG, "box dimension %d != workspace dimension %d", o->d, dw);
    return 0;
}

// The cell-ordered copy of the last grid build, while it describes the samples' current shard (cleared by every
// other builder that reuses those buffers and by a change of the query range).
static CellOrder cell_order(const mpb200_samples *s) {
    if (!s || !s->pt_order_valid) return CellOrder{nullptr, nullptr, nullptr};
    return CellOrder{s->sorted_pos.as<double>(), (s->q1 - s->q0 != s->N) ? s->q_order.as<int>() : nullptr,
                     s->pt_order.as<int>()};
}

int points_free_device(const double *dV, int64_t n, int d, const mpb200_obstacles *o, const mpb200_space_desc *ss,
                       uint32_t *d_bits32, uint8_t *d_bytes, const mpb200_samples *cs) {
    SpaceDev S;
    int dw = 0;
    if (int rc = make_space(ss, d, &S, &dw)) return rc;
    if (int rc = check_obstacles(o, dw)) return rc;
    LaunchCfg L = make_cfg(o, n);
    const CellOrder co = cell_order(cs);
    cudaStream_t st = ctx().stream;
#define CALL(N_, DW_, K_)                                                                              \
    do {                                                                                               \
        if (int rc = prep_kernel(points_free_kernel<N_, DW_, K_>, L.smem)) return rc;                  \
        if (int rc = resident_grid(points_free_kernel<N_, DW_, K_>, L.smem, n, &L.grid)) return rc;    \
        points_free_kernel<N_, DW_, K_><<<L.grid, kThreads, L.smem, st>>>(dV, n, S, L.table, L.words, L.M, \
                                                                          L.use_smem, d_bits32, d_bytes, co); \
    } while (0)
    MPB_DISPATCH_DIMS(S.n, dw, o->kind, CALL);
#undef CALL
    MPB_LAUNCHED();
    return 0;
}

int edges_free_device(const mpb200_samples *s, mpb200_table *t, const mpb200_obstacles *o,
                      const mpb200_space_desc *ss, uint32_t *d_bits32, unsigned long long *d_counters) {
    SpaceDev S;
    int dw = 0;
    if (int rc = make_space(ss, s->d, &S, &dw)) return rc;
    if (int rc = check_obstacles(o, dw)) return rc;
    const double *dV = s->V.as<double>();
    const int64_t *colptr = t->colptr.as<int64_t>();
    const int64_t *rowval = t->rowval.as<int64_t>();
    LaunchCfg L = make_cfg(o, t->ncols);
    cudaStream_t st = ctx().stream;
    static const bool no_classify = getenv("MPB200_NO_CLASSIFY") != nullptr;
    const bool classify = t->euclid && S.s2w_kind == 0 && t->ncols > 0 && t->ncols < INT_MAX && !no_classify &&
                          (o->kind == 0 ? dw == 2 : (dw >= 2 && dw <= 10));
    if (classify) {  // one lane per column, then one warp per column of the list
        if (int rc = t->col_list.reserve(sizeof(int) * (size_t)(t->ncols + 1))) return rc;
        const CellOrder co = (t->has_order && t->grid_build == s->grid_build) ? cell_order(s) : CellOrder{nullptr, nullptr, nullptr};
        const int *order = t->has_order ? t->col_order.as<int>() : nullptr;
        int *list = t->col_list.as<int>();
#define CALLC(DW_, K_)                                                                                         \
        do {                                                                                                   \
            if (int rc = prep_kernel(classify_columns<DW_, K_>, L.smem)) return rc;                            \
            if (int rc = resident_grid(classify_columns<DW_, K_>, L.smem, t->ncols, &L.grid)) return rc;       \
            classify_columns<DW_, K_><<<L.grid, kThreads, L.smem, st>>>(dV, colptr, t->ncols, t->col0, t->r, S, \
                                                                        L.table, L.words, L.M, L.use_smem, order, \
                                                                        co, d_bits32, d_counters, list);       \
            MPB_LAUNCHED();                                                                                    \
            if (int rc = prep_kernel(edges_free_kernel<DW_, DW_, K_>, L.smem)) return rc;                      \
            if (int rc = resident_grid(edges_free_kernel<DW_, DW_, K_>, L.smem, t->ncols * 32, &L.grid)) return rc; \
            edges_free_kernel<DW_, DW_, K_><<<L.grid, kThreads, L.smem, st>>>(dV, colptr, rowval, t->ncols, t->col0, \
                                                                              S, L.table, L.words, L.M, L.use_smem, \
                                                                              d_bits32, d_counters, list,      \
                                                                              d_counters + 1);                 \
        } while (0)
        if (o->kind == 0) {
            CALLC(2, 0);
        } else {
            switch (dw) {
            case 2: CALLC(2, 1); break; case 3: CALLC(3, 1); break; case 4: CALLC(4, 1); break;
            case 5: CALLC(5, 1); break; case 6: CALLC(6, 1); break; case 7: CALLC(7, 1); break;
            case 8: CALLC(8, 1); break; case 9: CALLC(9, 1); break; default: CALLC(10, 1); break;
            }
        }
#undef CALLC
        MPB_LAUNCHED();
        return 0;
    }
    // one warp per column
#define CALL(N_, DW_, K_)                                                                                  \
    do {                                                                                                   \
        if (int rc = prep_kernel(edges_free_kernel<N_, DW_, K_>, L.smem)) return rc;                       \
        if (int rc = resident_grid(edges_free_kernel<N_, DW_, K_>, L.smem, t->ncols * 32, &L.grid)) return rc; \
        edges_free_kernel<N_, DW_, K_><<<L.grid, kThreads, L.smem, st>>>(dV, colptr, rowval, t->ncols, t->col0, S, \
                                                                         L.table, L.words, L.M, L.use_smem, \
                                                                         d_bits32, d_counters, nullptr, nullptr); \
    } while (0)
    MPB_DISPATCH_DIMS(S.n, dw, o->kind, CALL);
#undef CALL
    MPB_LAUNCHED();
    return 0;
}

int segments_free_device(const double *dA, const double *dB, int64_t n, int d, const mpb200_obstacles *o,
                         const mpb200_space_desc *ss, uint8_t *d_out) {
    SpaceDev S;
    int dw = 0;
    if (int rc = make_space(ss, d, &S, &dw)) return rc;
    if (int rc = check_obstacles(o, dw)) return rc;
    LaunchCfg L = make_cfg(o, n);
    cudaStream_t st = ctx().stream;
#define CALL(N_, DW_, K_)                                                                               \
    do {                                                                                                \
        if (int rc = prep_kernel(segments_free_kernel<N_, DW_, K_>, L.smem)) return rc;                 \
        segments_free_kernel<N_, DW_, K_><<<L.grid, kThreads, L.smem, st>>>(dA, dB, n, S, L.table, L.words, \
                                                                            L.M, L.use_smem, d_out);    \
    } while (0)
    MPB_DISPATCH_DIMS(S.n, dw, o->kind, CALL);
#undef CALL
    MPB_LAUNCHED();
    return 0;
}

// Fill dV (n_want x n states, AoS) with the first n_want free candidates of the stream; *h_used = candidates consumed.
// `scratch` holds two int arrays of the chunk size, `tmp` the scan sums.
int sample_free_device(const mpb200_obstacles *o, const mpb200_space_desc *ss, int64_t n_want, uint64_t seed,
                       double *dV, DevBuf &scratch, DevBuf &tmp, int64_t *h_used) {
    SpaceDev S;
    int dw = 0;
    if (int rc = make_space(ss, ss ? ss->n : 0, &S, &dw)) return rc;
    if (int rc = check_obstacles(o, dw)) return rc;
    Context &c = ctx();
    cudaStream_t st = c.stream;
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    int *d_total = reinterpret_cast<int *>(c.d_scalar + 12);  // free states in the chunk (upper half kept zero)
    long long *d_used = reinterpret_cast<long long *>(c.d_scalar + 13);
    MPB_CUDA(cudaMemsetAsync(d_used, 0, sizeof(long long), st));
    int64_t got = 0, c0 = 0, cands = 0, frees = 0;
    int empty_chunks = 0;
    *h_used = 0;
    while (got < n_want) {
        // chunk sized from the acceptance rate seen so far (first chunk: assume everything is free)
        const double p_hat = cands > 0 ? fmax((double)frees / (double)cands, 1e-3) : 1.0;
        int64_t C = (int64_t)((double)(n_want - got) * 1.1 / p_hat) + 4096;
        if (C > (int64_t(1) << 24)) C = int64_t(1) << 24;
        if (int rc = scratch.reserve(sizeof(int) * (size_t)(2 * C + 2))) return rc;
        if (int rc = tmp.reserve(sizeof(int64_t) * (size_t)(ceil_div(C, kScanTile) + 2))) return rc;
        int *flags = scratch.as<int>(), *offs = flags + C + 1;
        LaunchCfg L = make_cfg(o, C);
        MPB_CUDA(cudaMemsetAsync(d_total, 0, sizeof(int64_t), st));
#define CALLS(N_, DW_, K_)                                                                                     \
        do {                                                                                                       \
            if (int rc = prep_kernel(sample_flags_kernel<N_, DW_, K_>, L.smem)) return rc;                         \
            sample_flags_kernel<N_, DW_, K_><<<L.grid, kThreads, L.smem, st>>>(S, L.table, L.words, L.M, L.use_smem, \
                                                                               k0, k1, c0, C, flags);             \
            MPB_LAUNCHED();                                                                                        \
            if (int rc = exclusive_scan<int, int>(flags, C, offs, 0, tmp, d_total)) return rc;                     \
            sample_scatter_kernel<N_><<<L.grid, kThreads, 0, st>>>(S, k0, k1, c0, C, flags, offs, got, n_want, dV, \
                                                                   d_used);                                        \
        } while (0)
        MPB_DISPATCH_DIMS(S.n, dw, o->kind, CALLS);
#undef CALLS
        MPB_LAUNCHED();
        MPB_CUDA(cudaMemcpyAsync(c.h_scalar + 12, c.d_scalar + 12, sizeof(int64_t) * 2, cudaMemcpyDeviceToHost, st));
        MPB_CUDA(cudaStreamSynchronize(st));
        const int64_t total = c.h_scalar[12];
        got += total;
        frees += total;
        cands += C;
        c0 += C;
        empty_chunks = total ? 0 : empty_chunks + 1;
        if (empty_chunks >= 8)
            return fail(MPB200_EARG, "no free state among %lld candidates: the free space is empty", (long long)cands);
    }
    *h_used = c.h_scalar[13];
    return 0;
}

// ---- shortcutting planned paths, phase 1 (mpb200_shortcut_paths; shortcut.cu runs the minimum) ----------------------
// Row b of a path holds free(a, b) = motion_free(node a, node b) for every a < b.  One warp per row: node b's workspace
// image stays in registers while the lanes take the nodes a < b 32 at a time (coalesced), with the warp-collective
// segment test of column_edges; each ballot is one whole word of the row (a0 is a multiple of 32), so no atomics and no
// memset.  The rows of every path form one flat list (global row = global node) dealt to the warps of a resident grid in
// turn, so long and short paths share the warps.  Segment tests are summed per warp and flushed with one atomicAdd per
// path the warp leaves.
template <int N, int DW, int KIND>
__global__ void __launch_bounds__(kThreads, (KIND == 0 || DW <= 4) ? 2 : 1)
shortcut_visibility_kernel(const ShortcutPath *__restrict__ paths, int npaths, int64_t nrows,
                           const double *__restrict__ nodes, SpaceDev S, const double *__restrict__ g_table,
                           int table_words, int M, bool use_smem, uint32_t *__restrict__ bits,
                           ShortcutResult *__restrict__ results) {
    extern __shared__ double s_table[];
    const double *T = stage_table(g_table, table_words, use_smem, s_table);
    const int lane = threadIdx.x & 31;
    const int64_t gwarp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    Obs2 O(KIND == 0 ? T : nullptr, KIND == 0);
    const LaneCull cl = lane_cull<KIND>(O);
    int cur = -1;
    unsigned long long my_checks = 0;  // lane 0: segment tests of path `cur` not yet added
    for (int64_t g = gwarp; g < nrows; g += nwarps) {
        const int q = shortcut_path_of(paths, npaths, g);
        if (q != cur) {
            if (lane == 0 && my_checks) atomicAdd(&results[cur].checks, my_checks);
            my_checks = 0;
            cur = q;
        }
        const int64_t node0 = paths[q].node0, bit0 = paths[q].bit0;
        const int words = paths[q].words;
        const int b = (int)(g - node0);
        double w[N], qw[DW];
#pragma unroll
        for (int k = 0; k < N; ++k) w[k] = nodes[g * N + k];
        state2workspace<N, DW>(S, w, qw);  // the last waypoint is never bounds-checked (Q4)
        uint32_t *row = bits + bit0 + (int64_t)b * words;
        const double *pv = nodes + node0 * N;
        for (int a0 = 0; a0 < b; a0 += 32) {
            const int a = a0 + lane;
            bool run = false;
            double v[N], p[DW];
#pragma unroll
            for (int k = 0; k < N; ++k) v[k] = 0.0;
            if (a < b) {
#pragma unroll
                for (int k = 0; k < N; ++k) v[k] = pv[(int64_t)a * N + k];
                run = in_state_space<N>(S, v);  // statespaces.jl:155: in_state_space(wps[1]) && segment test
            }
            state2workspace<N, DW>(S, v, p);
            // warp-collective: every lane must make the call (no short-circuit on `run`)
            bool seg_free;
            if (KIND == 0)
                seg_free = !warp_line_colliding_2d(O, cl.xl, cl.xh, cl.yl, cl.yh, p[0], p[DW > 1 ? 1 : 0], qw[0],
                                                   qw[DW > 1 ? 1 : 0], run);
            else
                seg_free = warp_box_segment_free<DW>(T, M, p, qw, run);
            const unsigned m = __ballot_sync(0xffffffffu, run && seg_free);
            const unsigned ran = __ballot_sync(0xffffffffu, run);
            if (lane == 0) {
                row[a0 >> 5] = m;
                my_checks += (unsigned long long)__popc(ran);
            }
        }
    }
    if (lane == 0 && my_checks) atomicAdd(&results[cur].checks, my_checks);
}

// The checks mpb200_segments_free makes of the space and obstacles, without a launch.
int shortcut_check_space(const mpb200_obstacles *o, const mpb200_space_desc *ss, int d) {
    SpaceDev S;
    int dw = 0;
    if (int rc = make_space(ss, d, &S, &dw)) return rc;
    if (int rc = check_obstacles(o, dw)) return rc;
#define CALL(N_, DW_, K_) do {} while (0)
    MPB_DISPATCH_DIMS(S.n, dw, o->kind, CALL);
#undef CALL
    return 0;
}

int shortcut_visibility_device(const ShortcutPath *paths, int npaths, int64_t nodes_total, const double *nodes, int d,
                               const mpb200_obstacles *o, const mpb200_space_desc *ss, uint32_t *bits,
                               ShortcutResult *results) {
    SpaceDev S;
    int dw = 0;
    if (int rc = make_space(ss, d, &S, &dw)) return rc;
    if (int rc = check_obstacles(o, dw)) return rc;
    LaunchCfg L = make_cfg(o, nodes_total);
    cudaStream_t st = ctx().stream;
    static const int env_grid = [] { const char *e = getenv("MPB200_SHORTCUT_GRID"); return e ? atoi(e) : 0; }();
#define CALL(N_, DW_, K_)                                                                                        \
    do {                                                                                                         \
        if (int rc = prep_kernel(shortcut_visibility_kernel<N_, DW_, K_>, L.smem)) return rc;                    \
        if (int rc = resident_grid(shortcut_visibility_kernel<N_, DW_, K_>, L.smem, nodes_total * 32, &L.grid))  \
            return rc;                                                                                           \
        if (env_grid > 0 && (unsigned)env_grid < L.grid) L.grid = (unsigned)env_grid;                            \
        shortcut_visibility_kernel<N_, DW_, K_><<<L.grid, kThreads, L.smem, st>>>(                               \
            paths, npaths, nodes_total, nodes, S, L.table, L.words, L.M, L.use_smem, bits, results);             \
    } while (0)
    MPB_DISPATCH_DIMS(S.n, dw, o->kind, CALL);
#undef CALL
    MPB_LAUNCHED();
    return 0;
}

// lazy GMT*: step 4 runs motion_free (the segment test of segments_free_kernel) on the winning entry, on one lane
template <int N, int DW, int KIND>
struct GmtStraightEdge {
    static constexpr bool kLazy = true;
    SpaceDev S;
    const double *T;
    int M;
    __device__ bool operator()(const GmtArgs &a, long long, int y, int x, GmtCtl *ctl) const {
        double v[N], w[N];
        gmt_endpoints<N>(a, y, x, v, w);
        bool checked;
        const bool ok = motion_free<N, DW, KIND>(S, T, M, v, w, &checked);
        gmt_count_segments(ctl, checked ? 1 : 0);
        return ok;
    }
};

int gmt_lazy_straight(const GmtArgs &a, const mpb200_obstacles *o, const mpb200_space_desc *ss, int *blocks) {
    SpaceDev S;
    int dw = 0;
    if (int rc = make_space(ss, a.d, &S, &dw)) return rc;
    if (int rc = check_obstacles(o, dw)) return rc;
#define CALL(N_, DW_, K_) return gmt_launch(a, GmtStraightEdge<N_, DW_, K_>{S, o->table.as<double>(), o->M}, blocks)
    MPB_DISPATCH_DIMS(S.n, dw, o->kind, CALL);
#undef CALL
    return 0;
}

}  // namespace mpb
