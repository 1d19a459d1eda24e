// grid_rball.cu -- K1 (uniform-grid build) + K2 (r-ball count / fill) for d = 2, 3.
//
// Replaces helper_data_structures(V, ::Euclidean) = KDTree build (geometric.jl:14-15) and,
// for every query column, inball(V, dist, ::TreeDistanceDS, v, r) (nearneighbors.jl:179-183):
// member iff j != v and s = sum_i (V[v]_i - V[j]_i)^2 <= r*r, evaluated in index order
// with one rounding per operation (no FMA); stored value sqrt(s); rows ascending.
//
// Data layout in HBM: samples stay AoS (d x N column-major, exactly the reference's
// Vector{SVector{d,Float64}}); the grid adds a cell-ordered AoS copy + the permutation, so a
// 3-cell x-run of candidates is one contiguous span; three (d=2) or nine (d=3) x-runs per query.
// Pipeline of one build (the first five steps are one CUDA graph):
//   cell_histogram (each sample's cell + its rank in the cell) -> scan -> cell_scatter (no atomics)
//   [shard form: one pass over the samples that can be in range, compact list, query collection]
//   -> rball_count (thread per query in cell order; FP64 test; one byte per hit) -> colptr scan
//   -> nnz read-back (event) overlapped with rball_fill (per column: hit bytes -> index + point ->
//      distance -> register bitonic sort by index -> contiguous Int64/Float64 burst)
//   -> rball_fill_big / sort_big_columns for the rare columns beyond 64 entries or 255 candidates.
#include "common.cuh"
#include "predicates.cuh"
#include "scan.cuh"
#include <algorithm>
#include <cstdlib>

namespace mpb {

constexpr int kWarpsPerBlock = 8;
constexpr int kStageCap = 256;  // hits staged per warp; larger columns take the spill path

struct GridDev {
    double lo[3];
    double inv_h;
    int n[3];
    // only samples inside [in_lo, in_hi] are inserted: the query shard's bounding box grown by r.  With a
    // spatially coherent query range (samples stored in stripe / Morton order) each GPU then grids
    // only its stripe + halo instead of the whole replicated sample set.
    double in_lo[3], in_hi[3];
};

template <int D>
__device__ __forceinline__ void cell_of(const GridDev &g, const double *p, int *c) {
#pragma unroll
    for (int i = 0; i < D; ++i) {
        // explicit intrinsics: every kernel must compute the identical cell for a point
        double q = __dmul_rn(__dsub_rn(p[i], g.lo[i]), g.inv_h);
        int ci = (int)floor(q);
        ci = ci < 0 ? 0 : ci;
        ci = ci >= g.n[i] ? g.n[i] - 1 : ci;
        c[i] = ci;
    }
}
template <int D>
__device__ __forceinline__ int cell_linear(const GridDev &g, const int *c) {
    int l = c[D - 1];
#pragma unroll
    for (int i = D - 2; i >= 0; --i) l = l * g.n[i] + c[i];
    return l;
}

// one sample of an AoS array: a single 16-byte access for d = 2 (the arrays are 16-byte aligned)
template <int D>
__device__ __forceinline__ void load_point(const double *__restrict__ A, int64_t j, double *p) {
    if (D == 2) {
        const double2 v = reinterpret_cast<const double2 *>(A)[j];
        p[0] = v.x; p[D - 1] = v.y;
    } else {
#pragma unroll
        for (int i = 0; i < D; ++i) p[i] = A[j * D + i];
    }
}
template <int D>
__device__ __forceinline__ void store_point(double *__restrict__ A, int64_t j, const double *p) {
    if (D == 2) {
        reinterpret_cast<double2 *>(A)[j] = make_double2(p[0], p[D - 1]);
    } else {
#pragma unroll
        for (int i = 0; i < D; ++i) A[j * D + i] = p[i];
    }
}

// ---- bounding box ------------------------------------------------------------------
__global__ void __launch_bounds__(256) bbox_partial(const double *__restrict__ V, int64_t N, int d,
                                                    double *__restrict__ part /*grid x 2d*/) {
    __shared__ double smin[8][16], smax[8][16];
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    for (int i = 0; i < d; ++i) {
        double mn = inf, mx = -inf;
        for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < N; j += (int64_t)gridDim.x * blockDim.x) {
            double x = V[j * d + i];
            mn = fmin(mn, x);
            mx = fmax(mx, x);
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        }
        if ((threadIdx.x & 31) == 0) { smin[threadIdx.x >> 5][i] = mn; smax[threadIdx.x >> 5][i] = mx; }
    }
    __syncthreads();
    if (threadIdx.x < d) {
        double mn = inf, mx = -inf;
        for (int w = 0; w < 8; ++w) { mn = fmin(mn, smin[w][threadIdx.x]); mx = fmax(mx, smax[w][threadIdx.x]); }
        part[(size_t)blockIdx.x * 2 * d + threadIdx.x] = mn;
        part[(size_t)blockIdx.x * 2 * d + d + threadIdx.x] = mx;
    }
}
__global__ void bbox_final(const double *__restrict__ part, int nb, int d, double *__restrict__ out) {
    const int i = threadIdx.x >> 5, lane = threadIdx.x & 31;  // one warp per dimension
    if (i >= d) return;
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    double mn = inf, mx = -inf;
    for (int b = lane; b < nb; b += 32) { mn = fmin(mn, part[(size_t)b * 2 * d + i]); mx = fmax(mx, part[(size_t)b * 2 * d + d + i]); }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (lane == 0) { out[i] = mn; out[d + i] = mx; }
}

// ---- K1: grid build ------------------------------------------------------------------
// The histogram's atomicAdd already hands every sample its rank inside its cell: it is kept (packed with the
// cell id would not fit 32 bits, so a second int array), and the scatter needs neither atomics nor a zeroed
// cursor array.
template <int D>
__global__ void __launch_bounds__(256) cell_histogram(const double *__restrict__ V, int64_t N, GridDev g,
                                                      int *__restrict__ hist, int *__restrict__ cell_id,
                                                      int *__restrict__ cell_rank) {
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= N) return;
    double p[D];
    bool inside = true;
    load_point<D>(V, j, p);
#pragma unroll
    for (int i = 0; i < D; ++i) inside = inside && (p[i] >= g.in_lo[i] && p[i] <= g.in_hi[i]);
    if (!inside) { cell_id[j] = -1; return; }  // cannot be within r of any query of this shard
    int c[D];
    cell_of<D>(g, p, c);
    int l = cell_linear<D>(g, c);
    cell_id[j] = l;
    cell_rank[j] = atomicAdd(&hist[l], 1);
}
template <int D>
__global__ void __launch_bounds__(256) cell_scatter(const double *__restrict__ V, int64_t N,
                                                    const int *__restrict__ cell_id, const int *__restrict__ cell_rank,
                                                    const int *__restrict__ cell_start,
                                                    int *__restrict__ sorted_idx, double *__restrict__ sorted_pos) {
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= N) return;
    int l = cell_id[j];
    if (l < 0) return;
    int pos = cell_start[l] + cell_rank[j];
    sorted_idx[pos] = (int)j;
    double p[D];
    load_point<D>(V, j, p);
    store_point<D>(sorted_pos, pos, p);
}

// number of adjacent pairs out of order along the first coordinate (0 <=> sorted)
__global__ void __launch_bounds__(256) count_x_inversions(const double *__restrict__ V, int64_t N, int d,
                                                          int *__restrict__ n_bad) {
    bool bad = false;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j + 1 < N; j += (int64_t)gridDim.x * blockDim.x)
        bad = bad || !(V[j * d] <= V[(j + 1) * d]);
    if (__syncthreads_or(bad) && threadIdx.x == 0) atomicAdd(n_bad, 1);
}
// x-sorted samples: the index range [lo, hi) whose first coordinate lies in [x_lo, x_hi].  Two warps, one per
// bound, each a 32-ary search (32 probes per step, ballot): 5 dependent loads for 8M samples instead of 23.
__global__ void __launch_bounds__(64) stripe_range(const double *__restrict__ V, int64_t N, int d, double x_lo,
                                                   double x_hi, long long *__restrict__ range) {
    const int lane = threadIdx.x & 31, upper = threadIdx.x >> 5;
    if (V == nullptr) {  // unsorted samples: look at all of them
        if (lane == 0) range[upper] = upper ? N : 0;
        return;
    }
    // first index whose x is NOT below the bound: "x < x_lo" for the lower end, "x <= x_hi" for the upper end
    int64_t lo = 0, hi = N;
    while (lo < hi) {
        const int64_t step = (hi - lo + 31) >> 5;
        const int64_t j = lo + lane * step;
        const bool below = j < hi && (upper ? (V[j * d] <= x_hi) : (V[j * d] < x_lo));
        const int c = __popc(__ballot_sync(0xffffffffu, below));  // probes are monotone: c ones, then zeros
        if (c == 0) { hi = lo; break; }
        const int64_t nlo = lo + (int64_t)(c - 1) * step + 1;
        const int64_t nhi = lo + (int64_t)c * step;
        lo = nlo;
        hi = nhi < hi ? nhi : hi;
    }
    if (lane == 0) range[upper] = lo;
}

// Append slots for the threads of a 256-thread block whose `flag` is set: ONE atomicAdd on the list counter per block
// (same-address atomics serialise in L2; per-warp aggregation was measured at ~30 us per million items).  Returns
// the thread's slot (valid when flag).  All threads of the block must call it.
__device__ __forceinline__ int block_append_slot(bool flag, int *__restrict__ counter) {
    __shared__ int s_warp[8];
    __shared__ int s_base;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const unsigned m = __ballot_sync(0xffffffffu, flag);
    if (lane == 0) s_warp[wid] = __popc(m);
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) { const int c = s_warp[w]; s_warp[w] = tot; tot += c; }
        s_base = tot ? atomicAdd(counter, tot) : 0;
    }
    __syncthreads();
    return s_base + s_warp[wid] + __popc(m & ((1u << lane) - 1u));
}

template <int D>
__global__ void __launch_bounds__(256) cell_histogram_shard(const double *__restrict__ V, GridDev g,
                                                            const long long *__restrict__ range,
                                                            int *__restrict__ hist, int *__restrict__ in_j,
                                                            int *__restrict__ in_l, int *__restrict__ in_r,
                                                            int *__restrict__ n_in) {
    // samples [range[0], range[1]): everything, or -- for x-sorted samples -- only the stripe that can be in range
    const int64_t j_lo = range[0], j_hi = range[1];
    for (int64_t b0 = j_lo + (int64_t)blockIdx.x * blockDim.x; b0 < j_hi; b0 += (int64_t)gridDim.x * blockDim.x) {  // block-uniform
        const int64_t j = b0 + threadIdx.x;
        bool inside = j < j_hi;
        double p[D];
        if (inside) {
#pragma unroll
            for (int i = 0; i < D; ++i) {
                p[i] = V[j * D + i];
                inside = inside && (p[i] >= g.in_lo[i] && p[i] <= g.in_hi[i]);
            }
        }
        int l = -1, rank = 0;
        if (inside) {
            int c[D];
            cell_of<D>(g, p, c);
            l = cell_linear<D>(g, c);
            rank = atomicAdd(&hist[l], 1);  // the sample's rank inside its cell: the scatter needs no atomics
        }
        const int slot = block_append_slot(inside, n_in);
        if (inside) {
            in_j[slot] = (int)j;
            in_l[slot] = l;
            in_r[slot] = rank;
        }
        __syncthreads();  // block_append_slot's shared scratch is reused by the next chunk
    }
}
template <int D>
__global__ void __launch_bounds__(256) cell_scatter_shard(const double *__restrict__ V, const int *__restrict__ n_in,
                                                          const int *__restrict__ in_j, const int *__restrict__ in_l,
                                                          const int *__restrict__ in_r, const int *__restrict__ cell_start,
                                                          int *__restrict__ sorted_idx, double *__restrict__ sorted_pos) {
    const int n = *n_in;  // grid-stride: the grid is sized for the SMs, not for the (device-side) list length
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int j = in_j[i];
        const int pos = cell_start[in_l[i]] + in_r[i];
        sorted_idx[pos] = j;
        double p[D];
        load_point<D>(V, j, p);
        store_point<D>(sorted_pos, pos, p);
    }
}
__global__ void __launch_bounds__(256) collect_queries(const int *__restrict__ sorted_idx, const int *__restrict__ n_in,
                                                       int64_t q0, int64_t q1, int *__restrict__ q_order,
                                                       int *__restrict__ n_q) {
    const int n = *n_in;
    for (int64_t b0 = (int64_t)blockIdx.x * blockDim.x; b0 < n; b0 += (int64_t)gridDim.x * blockDim.x) {  // block-uniform
        const int64_t k = b0 + threadIdx.x;
        const bool mine = k < n && sorted_idx[k] >= q0 && sorted_idx[k] < q1;
        const int slot = block_append_slot(mine, n_q);
        if (mine) q_order[slot] = (int)k;
        __syncthreads();  // block_append_slot's shared scratch is reused by the next chunk
    }
}

// ---- K2: r-ball ------------------------------------------------------------------------
// squared distance in the reference's order: s = (a1-b1)^2; s = s + (a_i-b_i)^2 ...
template <int D>
__device__ __forceinline__ double sqdist(const double *a, const double *b) {
    double t = __dsub_rn(a[0], b[0]);
    double s = __dmul_rn(t, t);
#pragma unroll
    for (int i = 1; i < D; ++i) {
        t = __dsub_rn(a[i], b[i]);
        s = __dadd_rn(s, __dmul_rn(t, t));
    }
    return s;
}

// Enumerate the candidate span [beg, end) of x-run `run` (0 .. 3^(D-1)-1) around cell c.
template <int D>
__device__ __forceinline__ bool run_span(const GridDev &g, const int *c, int run, const int *__restrict__ cell_start,
                                         int *beg, int *end) {
    int cc[D];
    cc[0] = 0;
    int rr = run;
#pragma unroll
    for (int i = 1; i < D; ++i) {
        int dlt = rr % 3 - 1;
        rr /= 3;
        cc[i] = c[i] + dlt;
        if (cc[i] < 0 || cc[i] >= g.n[i]) return false;
    }
    int x0 = c[0] > 0 ? c[0] - 1 : 0;
    int x1 = c[0] + 1 < g.n[0] ? c[0] + 1 : g.n[0] - 1;
    cc[0] = x0;
    int l0 = cell_linear<D>(g, cc);
    *beg = cell_start[l0];
    *end = cell_start[l0 + (x1 - x0) + 1];
    return true;
}

// ---- thread-per-query passes -------------------------------------------------------------
// Queries are visited in CELL order (one thread per query), so the 32 lanes of a warp sit in the
// same or adjacent cells and read the same candidate spans (broadcast / L1 hits), and every
// lane is busy.  q_order (optional) lists the cell-order positions owned by this shard.
constexpr int kQThreads = 64;                 // two warps per block: measured 1% faster than 128 (less tail, finer balance)
constexpr int kListCap = 64;                  // hits staged per query thread; more -> warp path

constexpr int kMaxCand = 255;  // candidates per query addressable by the one-byte hit list

// candidate spans of a query: begs[r], lens[r] for the 3^(D-1) x-runs (len 0 = outside the grid)
template <int D>
__device__ __forceinline__ int query_spans(const GridDev &g, const double *p, const int *__restrict__ cell_start,
                                           int *begs, int *lens) {
    constexpr int kRuns = (D == 2) ? 3 : 9;
    int c[D];
    cell_of<D>(g, p, c);
    int total = 0;
#pragma unroll
    for (int run = 0; run < kRuns; ++run) {
        int beg = 0, end = 0;
        if (!run_span<D>(g, c, run, cell_start, &beg, &end)) { beg = 0; end = 0; }
        begs[run] = beg;
        lens[run] = end - beg;
        total += end - beg;
    }
    return total;
}

// Count pass.  Besides the per-column count it records WHICH candidates hit: one byte per hit
// (the candidate's number in run order), staged per thread in shared memory and written out by
// the warp as a [tile = 32 queries][slot][lane] byte array (one 32-byte sector per slot), so the
// fill pass never re-evaluates a distance and reads its column's list with coalesced byte loads.
//
// The kernel is bound by the L1 data pipe (ncu r1k: l1tex__data_pipe_lsu_wavefronts 86% of peak): the
// lanes of a warp sit in 3-4 different cells, so every candidate load touches 3-4 lines.  Measured
// alternatives that did NOT help: an FP32 grid-relative prefilter with exact FP64 recheck in a rounding
// band (8-byte loads; count 96 -> 102 us, scatter +22 us for the extra array), staging the warp's union
// spans in shared memory (60 registers, 100 us), unroll 1/2/8 (+-2 us), and a cell-centric form (r1q: the warp takes
// one grid cell of its tile at a time, lanes hold the cell's candidates in registers, the cell's queries are
// broadcast one after the other, hits compacted by ballot + popc into 64-byte rows per query): no per-test loads
// and 32/32 lanes active, but the per-round bookkeeping (ballot, two popc, slot, byte store) doubles the warp
// instructions (122M against 60M) and the kernel becomes issue-bound at 83% -- 142 us; the per-query row layout
// also cost the fill 7% (its list reads were L1 hits shared by the 32 columns of a tile, now one cold line each).
template <int D>
__global__ void __launch_bounds__(kQThreads)
rball_count(const double *__restrict__ sorted_pos, const int *__restrict__ sorted_idx,
            const int *__restrict__ q_order, int64_t nq, int64_t q0, GridDev g, double r2,
            const int *__restrict__ cell_start, int list_cap, int *__restrict__ counts, int *__restrict__ col_order,
            int *__restrict__ pt_order, uint32_t *__restrict__ hit_lists, int *__restrict__ big_list, unsigned long long *__restrict__ n_big) {
    constexpr int kRuns = (D == 2) ? 3 : 9;
    __shared__ __align__(16) unsigned char s_hits[kListCap][kQThreads];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int cnt = 0;
    if (t < nq) {
        const int pos = q_order ? q_order[t] : (int)t;
        double p[D];
#pragma unroll
        for (int i = 0; i < D; ++i) p[i] = sorted_pos[(size_t)pos * D + i];
        int begs[kRuns], lens[kRuns];
        const int total = query_spans<D>(g, p, cell_start, begs, lens);
        int j = 0;
#pragma unroll
        for (int run = 0; run < kRuns; ++run) {
            const int beg = begs[run], end = begs[run] + lens[run];
            // branch-free body (predicated store), unrolled: the loads of several candidates are in flight
#pragma unroll 4
            for (int k = beg; k < end; ++k) {
                double b[D];
                if (D == 2) {
                    const double2 v = reinterpret_cast<const double2 *>(sorted_pos)[k];  // one 16-byte load
                    b[0] = v.x; b[D - 1] = v.y;
                } else {
#pragma unroll
                    for (int i = 0; i < D; ++i) b[i] = sorted_pos[(size_t)k * D + i];
                }
                const bool hit = (k != pos) & (sqdist<D>(p, b) <= r2);
                if (hit & (cnt < kListCap)) s_hits[cnt][threadIdx.x] = (unsigned char)(j + (k - beg));
                cnt += hit ? 1 : 0;
            }
            j += end - beg;
        }
        const int w = (int)(sorted_idx[pos] - q0);
        counts[w] = cnt;
        col_order[t] = w;  // columns in cell order, for the collision passes (classify_columns)
        pt_order[t] = w;   // the same permutation kept with the sample set (points_free_kernel)
        if (cnt > 0 && (cnt > list_cap || total > kMaxCand)) {
            unsigned long long slot = atomicAdd(n_big, 1ULL);
            big_list[slot] = w;
        }
    }
    // warp writes its tile: slot rows 0 .. max(cnt)-1, four rows (8 words each) per step
    int kmax = min(cnt, kListCap);
#pragma unroll
    for (int o = 16; o; o >>= 1) kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, o));
    __syncwarp();
    const int64_t tile = (int64_t)blockIdx.x * (kQThreads / 32) + wid;
    for (int n0 = 0; n0 < kmax; n0 += 4) {
        const int n = n0 + (lane >> 3);
        if (n < kmax) {
            const uint32_t word = reinterpret_cast<const uint32_t *>(&s_hits[n][wid * 32])[lane & 7];
            hit_lists[(tile * kListCap + n) * 8 + (lane & 7)] = word;
        }
    }
}

// ascending bitonic sort of two keys per lane (element e = lane + 32 r)
__device__ __forceinline__ void bitonic64(unsigned &k0, unsigned &k1, int lane) {
#pragma unroll
    for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            const unsigned o0 = __shfl_xor_sync(0xffffffffu, k0, stride);
            const unsigned o1 = __shfl_xor_sync(0xffffffffu, k1, stride);
            const bool lower = (lane & stride) == 0;
            const bool up0 = (lane & size) == 0;                 // element lane
            const bool up1 = ((lane + 32) & size) == 0;          // element lane + 32
            k0 = (lower == up0) ? min(k0, o0) : max(k0, o0);
            k1 = (lower == up1) ? min(k1, o1) : max(k1, o1);
        }
    }
    {   // size 64, stride 32: register-local, ascending
        const unsigned lo = min(k0, k1), hi = max(k0, k1);
        k0 = lo; k1 = hi;
    }
#pragma unroll
    for (int stride = 16; stride > 0; stride >>= 1) {
        const unsigned o0 = __shfl_xor_sync(0xffffffffu, k0, stride);
        const unsigned o1 = __shfl_xor_sync(0xffffffffu, k1, stride);
        const bool lower = (lane & stride) == 0;
        k0 = lower ? min(k0, o0) : max(k0, o0);
        k1 = lower ? min(k1, o1) : max(k1, o1);
    }
}

// Fill.  Thread t owns query t of the cell order and parks that query's record (point, column
// base, candidate spans) in shared memory; the warp then walks over its 32 columns, U at a time,
// reading the record of the current column with a few broadcast 16-byte loads (no shuffles, and
// the record does not occupy registers).  For a column, lane e reads the e-th byte of the
// column's hit list (written by rball_count), maps the candidate number to a cell-order
// position, and loads the sample index AND the neighbour position together (independent loads
// from the cache-friendly cell-ordered copy); the exact distance is recomputed there and parked
// in shared memory by source slot.  The column is then sorted by index with a register bitonic
// network over the lanes (key = index << 6 | source slot), each lane picks up the distance of
// its sorted entry from the slot named in the key, and the column is written as one contiguous
// Int64/Float64 burst.  Columns with more than kListCap entries or more than kMaxCand
// candidates are left to rball_fill_big.  Requires N < 2^26 (key packing).
//
// Measured alternatives: (r1o) prefetching the next column group's hit byte -> position -> index/point chain
// one group ahead (software pipeline) changed nothing (297 us for U = 1, 2, 4): the kernel is bound by LSU
// wavefronts + issue slots, not by the latency of that chain, although half the stall samples sit on it.
// Visiting the tile's columns longest-first (so that groups needing the 64-key network cluster): fill 288 -> 320 us.
// (r1m) ranking each index against the column's indices read back from
// shared memory four at a time (no shuffles, rows stored at base + rank) halves the LSU
// wavefronts of the sort but costs ~2.3 ALU instructions per comparison: 269M warp
// instructions instead of 195M, issue-bound at 79%, 321 us against 295 us for this form.
// U = columns sorted concurrently by one warp (independent dependency chains vs register budget)
template <int D, int U>
__global__ void __launch_bounds__(kQThreads)
rball_fill(const double *__restrict__ sorted_pos, const int *__restrict__ sorted_idx,
           const int *__restrict__ q_order, const unsigned char *__restrict__ hit_lists, int64_t nq, int64_t q0,
           GridDev g, const int *__restrict__ cell_start, const int64_t *__restrict__ colptr,
           int64_t *__restrict__ rowval, double *__restrict__ nzval, const int64_t *__restrict__ nnz_dev,
           int64_t capacity) {
    // speculative launch (before the host has read nnz back): do nothing if the table would not fit
    // the buffers kept from the previous build; the host then grows them and launches again
    if (nnz_dev && *nnz_dev > capacity) return;
    constexpr int kRuns = (D == 2) ? 3 : 9;
    constexpr int kWBase = 2 * D, kWBeg = 2 * D + 2, kWLen = kWBeg + kRuns;  // word offsets in a record
    constexpr int NV = (kWLen + kRuns + 3) / 4;                                // 16-byte vectors per record
    __shared__ int4 s_rec[NV][kQThreads];
    __shared__ double s_dist[kQThreads / 32][U][kListCap];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned char *tile_list = hit_lists + (t >> 5) * (int64_t)(kListCap * 32);  // same tiling as rball_count
    int k_mine = 0;
    {
        int rec[NV * 4];
#pragma unroll
        for (int i = 0; i < NV * 4; ++i) rec[i] = 0;
        if (t < nq) {
            const int pos = q_order ? q_order[t] : (int)t;
            double p[D];
#pragma unroll
            for (int i = 0; i < D; ++i) {
                p[i] = sorted_pos[(size_t)pos * D + i];
                rec[2 * i] = __double2loint(p[i]);
                rec[2 * i + 1] = __double2hiint(p[i]);
            }
            const int64_t w = sorted_idx[pos] - q0;
            const long long base = colptr[w] - 1;
            rec[kWBase] = (int)(unsigned)(base & 0xffffffffLL);
            rec[kWBase + 1] = (int)(base >> 32);
            k_mine = (int)(colptr[w + 1] - colptr[w]);
            const int total = query_spans<D>(g, p, cell_start, rec + kWBeg, rec + kWLen);
            if (k_mine > kListCap || total > kMaxCand) k_mine = 0;  // handled by rball_fill_big
        }
#pragma unroll
        for (int v = 0; v < NV; ++v) s_rec[v][threadIdx.x] = make_int4(rec[4 * v], rec[4 * v + 1], rec[4 * v + 2], rec[4 * v + 3]);
    }
    __syncwarp();
    for (int cl0 = 0; cl0 < 32; cl0 += U) {
        int kc[U];
        unsigned key[U][2];
        int kmax = 0;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            kc[u] = __shfl_sync(0xffffffffu, k_mine, cl0 + u);
            kmax = max(kmax, kc[u]);
        }
        if (kmax == 0) continue;
        const int rounds = (kmax > 32) ? 2 : 1;  // warp-uniform
#pragma unroll
        for (int u = 0; u < U; ++u) {
            int rec[NV * 4];
#pragma unroll
            for (int v = 0; v < NV; ++v) {   // broadcast reads of column (cl0 + u)'s record
                const int4 q = s_rec[v][wid * 32 + cl0 + u];
                rec[4 * v] = q.x; rec[4 * v + 1] = q.y; rec[4 * v + 2] = q.z; rec[4 * v + 3] = q.w;
            }
            double pc[D];
#pragma unroll
            for (int i = 0; i < D; ++i) pc[i] = __hiloint2double(rec[2 * i + 1], rec[2 * i]);
            // element e = lane + 32 h: candidate number -> cell-order position -> sort key, distance
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                key[u][h] = 0xffffffffu;
                const int e = lane + 32 * h;
                if (h < rounds && e < kc[u]) {
                    int j = tile_list[e * 32 + cl0 + u];  // candidate number of the e-th hit of this column
                    int kp = 0;
#pragma unroll
                    for (int r = 0; r < kRuns; ++r) {  // run containing candidate j
                        const bool here = (j >= 0) && (j < rec[kWLen + r]);
                        kp = here ? rec[kWBeg + r] + j : kp;
                        j = here ? -1 : j - rec[kWLen + r];
                    }
                    const unsigned idx = (unsigned)sorted_idx[kp];
                    double b[D];
                    if (D == 2) {
                        const double2 v = reinterpret_cast<const double2 *>(sorted_pos)[kp];  // one 16-byte load
                        b[0] = v.x; b[D - 1] = v.y;
                    } else {
#pragma unroll
                        for (int i = 0; i < D; ++i) b[i] = sorted_pos[(size_t)kp * D + i];
                    }
                    key[u][h] = (idx << 6) | (unsigned)e;
                    s_dist[wid][u][e] = sqrt(sqdist<D>(pc, b));
                }
            }
        }
        __syncwarp();
        if (rounds == 1) {
#pragma unroll
            for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
                for (int stride = size >> 1; stride > 0; stride >>= 1) {
                    const bool up = (lane & size) == 0;
                    const bool lower = (lane & stride) == 0;
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const unsigned other = __shfl_xor_sync(0xffffffffu, key[u][0], stride);
                        key[u][0] = (lower == up) ? min(key[u][0], other) : max(key[u][0], other);
                    }
                }
            }
        } else {
#pragma unroll
            for (int u = 0; u < U; ++u) bitonic64(key[u][0], key[u][1], lane);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int2 bw = reinterpret_cast<const int2 *>(&s_rec[kWBase / 4][wid * 32 + cl0 + u])[(kWBase % 4) / 2];
            const long long basec = ((long long)bw.y << 32) | (unsigned)bw.x;
            const int ru = (kc[u] > 32) ? 2 : (kc[u] > 0 ? 1 : 0);  // warp-uniform
            for (int h = 0; h < ru; ++h) {
                const int e = lane + 32 * h;
                const unsigned ky = h ? key[u][1] : key[u][0];
                if (e < kc[u]) {  // streaming stores: the table is not read again by this kernel
                    __stcs(reinterpret_cast<long long *>(rowval) + basec + e, (long long)(ky >> 6) + 1);
                    __stcs(nzval + basec + e, s_dist[wid][u][ky & 63u]);  // distance parked by the entry's source slot
                }
            }
        }
        __syncwarp();  // s_dist is reused by the next group of columns
    }
}

// Warp-per-query path for the (rare) columns with more than kListCap hits, driven by big_list:
// hits are ballot-compacted into a per-warp stage and rank-sorted there (<= kStageCap), or
// spilled unsorted for sort_big_columns.
template <int D>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
rball_fill_big(const double *__restrict__ V, const int *__restrict__ big_list, int64_t n_big, int64_t q0, GridDev g,
               double r2, const int *__restrict__ cell_start, const int *__restrict__ sorted_idx,
               const double *__restrict__ sorted_pos, const int64_t *__restrict__ colptr,
               int64_t *__restrict__ rowval, double *__restrict__ nzval,
               int64_t *__restrict__ spill_row, double *__restrict__ spill_val) {
    constexpr int kRuns = (D == 2) ? 3 : 9;
    __shared__ int s_idx[kWarpsPerBlock][kStageCap];
    __shared__ double s_sq[kWarpsPerBlock][kStageCap];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t bi = (int64_t)blockIdx.x * kWarpsPerBlock + wid;
    if (bi >= n_big) return;
    const int64_t w = big_list[bi];
    const int64_t v = q0 + w;
    const int64_t base = colptr[w] - 1;
    const int k_total = (int)(colptr[w + 1] - colptr[w]);
    const bool big = k_total > kStageCap;  // warp-uniform
    double p[D];
#pragma unroll
    for (int i = 0; i < D; ++i) p[i] = V[v * D + i];
    int c[D];
    cell_of<D>(g, p, c);
    int n_hit = 0;
#pragma unroll
    for (int run = 0; run < kRuns; ++run) {
        int beg, end;
        if (!run_span<D>(g, c, run, cell_start, &beg, &end)) continue;
        for (int k0 = beg; k0 < end; k0 += 32) {
            int k = k0 + lane;
            bool hit = false;
            int idx = 0;
            double s = 0;
            if (k < end) {
                double b[D];
#pragma unroll
                for (int i = 0; i < D; ++i) b[i] = sorted_pos[(size_t)k * D + i];
                idx = sorted_idx[k];
                s = sqdist<D>(p, b);
                hit = (idx != (int)v) && (s <= r2);
            }
            unsigned m = __ballot_sync(0xffffffffu, hit);
            int off = n_hit + __popc(m & ((1u << lane) - 1u));
            if (hit) {
                if (!big) {
                    s_idx[wid][off] = idx;
                    s_sq[wid][off] = s;
                } else {  // spill path: unsorted, sorted later by sort_big_columns
                    spill_row[base + off] = (int64_t)idx + 1;
                    spill_val[base + off] = sqrt(s);
                }
            }
            n_hit += __popc(m);
        }
    }
    if (big) return;
    __syncwarp();
    // rank sort by sample index (indices are distinct), then one contiguous burst per column
    for (int e = lane; e < n_hit; e += 32) {
        int mine = s_idx[wid][e];
        int rank = 0;
        for (int j = 0; j < n_hit; ++j) rank += (s_idx[wid][j] < mine) ? 1 : 0;
        rowval[base + rank] = (int64_t)mine + 1;
        nzval[base + rank] = sqrt(s_sq[wid][e]);
    }
}

// spill path: one block per over-sized column; rank sort from the unsorted spill copy
__global__ void __launch_bounds__(256)
sort_big_columns(const int *__restrict__ big_list, const int64_t *__restrict__ colptr,
                 const int64_t *__restrict__ spill_row, const double *__restrict__ spill_val,
                 int64_t *__restrict__ rowval, double *__restrict__ nzval) {
    __shared__ int64_t tile[256];
    const int w = big_list[blockIdx.x];
    const int64_t base = colptr[w] - 1;
    const int k = (int)(colptr[w + 1] - colptr[w]);
    if (k <= kStageCap) return;  // already sorted in shared memory by rball_fill_big
    for (int e0 = 0; e0 < k; e0 += 256) {
        int e = e0 + threadIdx.x;
        int64_t mine = (e < k) ? spill_row[base + e] : 0;
        int rank = 0;
        for (int t0 = 0; t0 < k; t0 += 256) {
            __syncthreads();
            if (t0 + (int)threadIdx.x < k) tile[threadIdx.x] = spill_row[base + t0 + threadIdx.x];
            __syncthreads();
            int lim = min(256, k - t0);
            for (int j = 0; j < lim; ++j) rank += (tile[j] < mine) ? 1 : 0;
        }
        if (e < k) {
            rowval[base + rank] = mine;
            nzval[base + rank] = spill_val[base + e];
        }
    }
}

// ---- host side ---------------------------------------------------------------------------
template <int D>
static int build_table(mpb200_samples *s, double r, mpb200_table *t) {
    Context &c = ctx();
    cudaStream_t st = c.stream;
    const int64_t N = s->N, nq = s->q1 - s->q0;
    const double *V = s->V.as<double>();

    // bounding box (host copy made at samples_create) -> grid geometry
    // grid over the query shard's bounding box grown by r (clipped to the samples' box)
    double bb[6];
    const double grow = r * (1.0 + 1e-6);
    for (int i = 0; i < D; ++i) {
        const double pad = grow + 4.5e-16 * fmax(fabs(s->h_qbbox[i]), fabs(s->h_qbbox[D + i]));
        bb[i] = fmax(s->h_bbox[i], s->h_qbbox[i] - pad);
        bb[D + i] = fmin(s->h_bbox[D + i], s->h_qbbox[D + i] + pad);
        if (!(bb[i] <= bb[D + i])) { bb[i] = s->h_bbox[i]; bb[D + i] = s->h_bbox[i]; }
    }
    GridDev g;
    const int max_per_dim = (D == 2) ? 4096 : 256;
    double ext_max = 0;
    for (int i = 0; i < D; ++i) ext_max = fmax(ext_max, bb[D + i] - bb[i]);
    // cell edge >= r(1+1e-6): two points within r are always in adjacent cells, rounding included
    double h = r * (1.0 + 1e-6);
    if (!(h > ext_max / max_per_dim)) h = ext_max / max_per_dim;
    if (!(h > 0)) h = 1.0;
    int64_t ncells = 1;
    for (int i = 0; i < D; ++i) {
        g.lo[i] = bb[i];
        double cnt = floor((bb[D + i] - bb[i]) / h) + 1.0;
        if (cnt > max_per_dim + 1) cnt = max_per_dim + 1;
        g.n[i] = (int)cnt;
        ncells *= g.n[i];
    }
    for (int i = D; i < 3; ++i) { g.lo[i] = 0; g.n[i] = 1; }
    g.inv_h = 1.0 / h;
    for (int i = 0; i < 3; ++i) { g.in_lo[i] = i < D ? bb[i] : 0; g.in_hi[i] = i < D ? bb[D + i] : 0; }

    // ---- reserve every buffer of the front half up front (nothing may allocate during graph capture)
    if (int rc = s->cell_start.reserve(sizeof(int) * (size_t)(ncells + 1))) return rc;
    if (int rc = s->cell_fill.reserve(sizeof(int) * (size_t)(ncells + 1))) return rc;
    if (int rc = s->sorted_idx.reserve(sizeof(int) * (size_t)(3 * N + 3))) return rc;  // + cell_id, cell_rank scratch
    if (int rc = s->sorted_pos.reserve(sizeof(double) * (size_t)(D * N + 1))) return rc;
    if (int rc = s->scan_tmp.reserve(sizeof(int64_t) * (size_t)(ceil_div(ncells > N ? ncells : N, kScanTile) + 2))) return rc;
    if (nq != N)  // shard: q_order | compact in-range list (sample, cell, rank in cell)
        if (int rc = s->q_order.reserve(sizeof(int) * (size_t)(4 * N + 5))) return rc;
    if (int rc = t->counts.reserve(sizeof(int) * (size_t)(2 * nq + 2))) return rc;
    if (int rc = t->colptr.reserve(sizeof(int64_t) * (size_t)(nq + 1))) return rc;
    if (int rc = t->masks.reserve((size_t)kListCap * 32 * (size_t)(ceil_div(nq, 32) + 1))) return rc;
    if (int rc = t->col_order.reserve(sizeof(int) * (size_t)(nq + 1))) return rc;
    if (int rc = s->pt_order.reserve(sizeof(int) * (size_t)(nq + 1))) return rc;
    s->pt_order_valid = false;
    s->grid_build = next_serial();
    t->has_order = false;
    int *hist = s->cell_fill.as<int>();
    int *cell_start = s->cell_start.as<int>();
    int *sorted_idx = s->sorted_idx.as<int>();
    int *cell_id = sorted_idx + N, *cell_rank = cell_id + N;
    double *sorted_pos = s->sorted_pos.as<double>();
    uint32_t *hit_lists = t->masks.as<uint32_t>();
    int *counts = t->counts.as<int>();
    int *big_list = counts + nq;
    unsigned long long *d_nbig = reinterpret_cast<unsigned long long *>(c.d_scalar + 1);
    const int *q_order = (nq != N) ? s->q_order.as<int>() : nullptr;
    const double r2 = r * r;
    const unsigned nbN = (unsigned)ceil_div(N > 0 ? N : 1, 256);
    const unsigned nbQ = (unsigned)ceil_div(nq > 0 ? nq : 1, kQThreads);
    // key packing in rball_fill needs N < 2^26; beyond that every non-empty column is "big"
    const int list_cap = (N < (int64_t(1) << 26)) ? kListCap : 0;

    // the front half: K1 (histogram, scan, scatter) [+ shard compaction] + count pass + colptr scan
    auto front = [&]() -> int {
        if (nq != N) {  // shard: one pass over all N samples, everything else over the in-range ones
            int *qo = s->q_order.as<int>();
            int *in_j = qo + N + 1, *in_l = in_j + N + 1, *in_r = in_l + N + 1;
            int *n_in = reinterpret_cast<int *>(c.d_scalar + 6);  // length of the compact list
            int *n_q = reinterpret_cast<int *>(c.d_scalar + 7);   // queries collected (== nq)
            const unsigned nbS = (unsigned)std::min<int64_t>(nbN, (int64_t)c.sm_count * 8);
            MPB_CUDA(cudaMemsetAsync(hist, 0, sizeof(int) * (size_t)(ncells + 1), st));
            MPB_CUDA(cudaMemsetAsync(n_in, 0, sizeof(int64_t) * 2, st));
            long long *range = reinterpret_cast<long long *>(c.d_scalar + 10);  // [first, last) sample to look at
            if (s->sorted_x) {
                stripe_range<<<1, 64, 0, st>>>(V, N, D, g.in_lo[0], g.in_hi[0], range);
                MPB_LAUNCHED();
            } else {
                stripe_range<<<1, 64, 0, st>>>(nullptr, N, D, 0.0, 0.0, range);  // whole array
                MPB_LAUNCHED();
            }
            cell_histogram_shard<D><<<nbS, 256, 0, st>>>(V, g, range, hist, in_j, in_l, in_r, n_in);
            MPB_LAUNCHED();
            if (int rc = exclusive_scan<int, int>(hist, ncells, cell_start, 0, s->scan_tmp, nullptr)) return rc;
            cell_scatter_shard<D><<<nbS, 256, 0, st>>>(V, n_in, in_j, in_l, in_r, cell_start, sorted_idx, sorted_pos);
            MPB_LAUNCHED();
            collect_queries<<<nbS, 256, 0, st>>>(sorted_idx, n_in, s->q0, s->q1, qo, n_q);
            MPB_LAUNCHED();
        } else {
            MPB_CUDA(cudaMemsetAsync(hist, 0, sizeof(int) * (size_t)(ncells + 1), st));
            cell_histogram<D><<<nbN, 256, 0, st>>>(V, N, g, hist, cell_id, cell_rank);
            MPB_LAUNCHED();
            if (int rc = exclusive_scan<int, int>(hist, ncells, cell_start, 0, s->scan_tmp, nullptr)) return rc;
            cell_scatter<D><<<nbN, 256, 0, st>>>(V, N, cell_id, cell_rank, cell_start, sorted_idx, sorted_pos);
            MPB_LAUNCHED();
        }
        MPB_CUDA(cudaMemsetAsync(c.d_scalar, 0, sizeof(int64_t) * 2, st));
        if (nq > 0) {
            rball_count<D><<<nbQ, kQThreads, 0, st>>>(sorted_pos, sorted_idx, q_order, nq, s->q0, g, r2, cell_start,
                                                     list_cap, counts, t->col_order.as<int>(), s->pt_order.as<int>(), hit_lists, big_list, d_nbig);
            MPB_LAUNCHED();
        }
        return exclusive_scan<int, int64_t>(counts, nq, t->colptr.as<int64_t>(), (int64_t)1, s->scan_tmp, c.d_scalar);
    };

    static const bool use_graph = getenv("MPB200_NO_GRAPH") == nullptr;
    phase_bank(MPB200_OP_TABLE);
    phase_mark(0);
    if (use_graph && nq > 0 && ncells > 0) {
        uint64_t key[32] = {};
        int kk = 0;
        auto put = [&](const void *p, size_t n) { uint64_t v = 0; memcpy(&v, p, n); key[kk++] = v; };
        const void *ptrs[] = {V, hist, cell_start, sorted_idx, sorted_pos, hit_lists, counts, t->colptr.p, s->scan_tmp.p,
                              s->q_order.p, c.d_scalar, (const void *)st, t->col_order.p, s->pt_order.p};
        for (const void *p : ptrs) put(&p, sizeof(p));
        put(&N, 8); put(&nq, 8); put(&s->q0, 8); put(&r, 8); put(&g.inv_h, 8); put(&g.lo[0], 8); put(&g.lo[1], 8);
        put(&g.lo[2], 8); put(&g.n[0], 4); put(&g.n[1], 4); put(&g.n[2], 4);
        put(&g.in_hi[0], 8); put(&g.in_hi[1], 8); put(&g.in_hi[2], 8);
        key[kk++] = (uint64_t)D;
        if (!(s->graph_exec && memcmp(key, s->graph_key, sizeof(key)) == 0)) {
            if (s->graph_exec) { cudaGraphExecDestroy(s->graph_exec); s->graph_exec = nullptr; }
            cudaGraph_t graph = nullptr;
            MPB_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
            const int64_t launches_before = c.launches;
            int rc = front();
            cudaError_t e = cudaStreamEndCapture(st, &graph);
            s->graph_launches = (int)(c.launches - launches_before);
            c.launches = launches_before;
            if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
            if (e != cudaSuccess) return fail(MPB200_ECUDA, "graph capture failed: %s", cudaGetErrorString(e));
            e = cudaGraphInstantiate(&s->graph_exec, graph, 0);
            cudaGraphDestroy(graph);
            if (e != cudaSuccess) { s->graph_exec = nullptr; return fail(MPB200_ECUDA, "graph instantiate failed: %s", cudaGetErrorString(e)); }
            memcpy(s->graph_key, key, sizeof(key));
        }
        MPB_CUDA(cudaGraphLaunch(s->graph_exec, st));
        c.launches += s->graph_launches;  // the kernels inside the graph still run
    } else {
        if (int rc = front()) return rc;
    }
    phase_mark(1);
    // sharded build attached to an exchange: the column lengths are final now -- they go out to the peers on a
    // side stream while this stream runs the fill and the validity kernels
    if (t->xchg && nq > 0)
        if (int rc = xchg_push_counts_early(t->xchg, t, t->colptr.as<int64_t>(), nq)) return rc;
    phase_mark(2);
    static const int fill_u = [] { const char *e = getenv("MPB200_FILL_U"); return e ? atoi(e) : 2; }();
    auto launch_fill = [&](const int64_t *guard, int64_t capacity) -> int {
        const int64_t *cp = t->colptr.as<int64_t>();
        int64_t *rv = t->rowval.as<int64_t>();
        double *nz = t->nzval.as<double>();
        const unsigned char *hl = t->masks.as<unsigned char>();
        if (fill_u == 4)
            rball_fill<D, 4><<<nbQ, kQThreads, 0, st>>>(sorted_pos, sorted_idx, q_order, hl, nq, s->q0, g, cell_start, cp, rv, nz, guard, capacity);
        else if (fill_u == 1)
            rball_fill<D, 1><<<nbQ, kQThreads, 0, st>>>(sorted_pos, sorted_idx, q_order, hl, nq, s->q0, g, cell_start, cp, rv, nz, guard, capacity);
        else
            rball_fill<D, 2><<<nbQ, kQThreads, 0, st>>>(sorted_pos, sorted_idx, q_order, hl, nq, s->q0, g, cell_start, cp, rv, nz, guard, capacity);
        MPB_LAUNCHED();
        return 0;
    };
    // Speculative fill: when the table still owns row/value buffers from an earlier build (a planner
    // rebuilding with a new radius, or repeated planning steps), the fill is enqueued BEFORE nnz is read
    // back, guarded on the device by nnz <= capacity, so the GPU does not idle during the read-back.
    static const bool no_spec = getenv("MPB200_NO_SPEC_FILL") != nullptr;
    const bool small_keys = N < (int64_t(1) << 26);
    const int64_t capacity = (int64_t)(std::min(t->rowval.cap / sizeof(int64_t), t->nzval.cap / sizeof(double))) - 1;
    const bool speculate = !no_spec && small_keys && nq > 0 && capacity > 0;
    // nnz and n_big come back right after the count scan; the host waits for THAT copy only (an event), so
    // with a speculative fill it learns nnz -- and returns to the caller, who can enqueue the validity passes --
    // while the fill is still running
    MPB_CUDA(cudaMemcpyAsync(c.h_scalar, c.d_scalar, sizeof(int64_t) * 2, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaEventRecord(c.ev_scalar, st));
    phase_mark(3);
    if (speculate) {
        if (int rc = launch_fill(c.d_scalar, capacity)) return rc;
        phase_mark(4);
    }
    MPB_CUDA(cudaEventSynchronize(c.ev_scalar));
    const int64_t nnz = c.h_scalar[0];
    const int64_t n_big = c.h_scalar[1];

    const bool filled = speculate && nnz <= capacity;
    if (int rc = t->rowval.reserve(sizeof(int64_t) * (size_t)(nnz + 1))) return rc;
    if (int rc = t->nzval.reserve(sizeof(double) * (size_t)(nnz + 1))) return rc;
    int64_t *spill_row = nullptr;
    double *spill_val = nullptr;
    if (n_big > 0) {
        if (int rc = t->scratch.reserve(16 * (size_t)(nnz + 1))) return rc;
        spill_row = t->scratch.as<int64_t>();
        spill_val = reinterpret_cast<double *>(spill_row + nnz);
    }
    if (!filled) phase_mark(3);
    if (nq > 0 && nnz > 0) {
        if (small_keys && !filled)
            if (int rc = launch_fill(nullptr, 0)) return rc;
        if (n_big > 0) {
            rball_fill_big<D><<<(unsigned)ceil_div(n_big, kWarpsPerBlock), kWarpsPerBlock * 32, 0, st>>>(
                V, big_list, n_big, s->q0, g, r2, cell_start, sorted_idx, sorted_pos, t->colptr.as<int64_t>(),
                t->rowval.as<int64_t>(), t->nzval.as<double>(), spill_row, spill_val);
            MPB_LAUNCHED();
            sort_big_columns<<<(unsigned)n_big, 256, 0, st>>>(big_list, t->colptr.as<int64_t>(), spill_row, spill_val,
                                                              t->rowval.as<int64_t>(), t->nzval.as<double>());
            MPB_LAUNCHED();
        }
    }
    if (!filled || n_big > 0) phase_mark(4);
    phases_collect(4);  // no trailing sync: the fill is stream-ordered before anything that reads the table
    t->ncols = nq;
    t->col0 = s->q0;
    t->nnz = nnz;
    t->r = r;
    t->euclid = true;
    t->has_order = nq > 0;
    t->grid_build = s->grid_build;
    s->pt_order_valid = nq > 0;
    return 0;
}

// bounding box of samples [j0, j1) into s->minmax (device); the caller copies it to the host
int compute_bbox(mpb200_samples *s, int64_t j0, int64_t j1) {
    Context &c = ctx();
    const int nb = 2 * c.sm_count;
    if (int rc = s->minmax.reserve(sizeof(double) * (size_t)(2 * s->d) * (size_t)(nb + 1))) return rc;
    double *out = s->minmax.as<double>();
    double *part = out + 2 * s->d;
    bbox_partial<<<nb, 256, 0, c.stream>>>(s->V.as<double>() + j0 * s->d, j1 - j0, s->d, part);
    MPB_LAUNCHED();
    bbox_final<<<1, 32 * s->d, 0, c.stream>>>(part, nb, s->d, out);
    MPB_LAUNCHED();
    return 0;
}

int check_sorted_x(mpb200_samples *s, int *d_flag) {
    Context &c = ctx();
    MPB_CUDA(cudaMemsetAsync(d_flag, 0, sizeof(int64_t), c.stream));
    count_x_inversions<<<2 * c.sm_count, 256, 0, c.stream>>>(s->V.as<double>(), s->N, s->d, d_flag);
    MPB_LAUNCHED();
    return 0;
}

int grid_inball_build(mpb200_samples *s, double r, mpb200_table *t) {
    if (s->d == 2) return build_table<2>(s, r, t);
    if (s->d == 3) return build_table<3>(s, r, t);
    return fail(MPB200_EARG, "grid r-ball supports d = 2, 3 (got %d)", s->d);
}

}  // namespace mpb
