// brute_rball.cu -- K3 + K4: Euclidean r-ball tables for d >= 4 (no useful spatial pruning: at the
// FMT* radius the ball spans a large part of the cube), as an all-pairs FP32 prefilter followed
// by the exact FP64 recheck of the few survivors.
//
// Replaces inball(V, dist, DS, v, r) over a KDTree / brute colwise distance
// (nearneighbors.jl:138-150,179-183; geometric.jl:4-6,14) for every query column.  Membership
// and stored distances are decided ONLY by the exact test  s = sum_i (V[v]_i - V[j]_i)^2 <= r*r
// (index order, one rounding per operation); the FP32 pass merely discards pairs that provably
// fail it: the threshold carries a rigorous bound on the FP32 conversion + accumulation error
// (derivation in DESIGN.md), so there are no false negatives.
//
// Layout: a padded FP32 AoS copy of the samples (float4 granules) is streamed through shared
// memory in tiles and read by broadcast; one thread owns one query column (its FP32 point in
// registers) and walks the samples in index order, so rows come out ascending and need no sort.
#include "common.cuh"
#include "scan.cuh"
#include "tc_rball.cuh"
#include <algorithm>
#include <cstdlib>

namespace mpb {

constexpr int kBrThreads = 256;
constexpr int kBrTile = 256;

template <int D>
__global__ void __launch_bounds__(256) to_float_padded(const double *__restrict__ V, int64_t N, float *__restrict__ Vf) {
    constexpr int DP = (D + 3) & ~3;
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= N) return;
#pragma unroll
    for (int i = 0; i < DP; ++i) Vf[j * DP + i] = (i < D) ? (float)V[j * D + i] : 0.0f;
}

template <int D>
__device__ __forceinline__ double exact_sq(const double *__restrict__ a, const double *__restrict__ b) {
    double t = __dsub_rn(a[0], b[0]);
    double s = __dmul_rn(t, t);
#pragma unroll
    for (int i = 1; i < D; ++i) {
        t = __dsub_rn(a[i], b[i]);
        s = __dadd_rn(s, __dmul_rn(t, t));
    }
    return s;
}

// MODE 0: count only; MODE 1: fill the CSC arrays (needs colptr); MODE 2: ONE sweep that counts and
// appends every hit (index, exact squared distance) to the query's slab of `cap` entries, so the
// all-pairs work is done once and a streaming compaction (slab_to_csc) finishes the table.
template <int D, int MODE>
__global__ void __launch_bounds__(kBrThreads)
brute_rball_kernel(const double *__restrict__ V, const float *__restrict__ Vf, int64_t N, int64_t q0, int64_t nq,
                   double r2, float thr32, int *__restrict__ counts, const int64_t *__restrict__ colptr,
                   int64_t *__restrict__ rowval, double *__restrict__ nzval, int cap, int *__restrict__ slab_j,
                   double *__restrict__ slab_s) {
    constexpr bool FILL = (MODE == 1);
    constexpr int DP = (D + 3) & ~3;
    __shared__ float4 tile[kBrTile * DP / 4];
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = w < nq;
    const int64_t q = q0 + w;
    float xq[DP];
#pragma unroll
    for (int i = 0; i < DP; ++i) xq[i] = active ? Vf[q * DP + i] : 0.0f;
    int cnt = 0;
    int64_t pos = (FILL && active) ? colptr[w] - 1 : 0;
    for (int64_t t0 = 0; t0 < N; t0 += kBrTile) {
        const int n_t = (int)((N - t0 < kBrTile) ? (N - t0) : kBrTile);
        __syncthreads();
        {
            const float4 *src = reinterpret_cast<const float4 *>(Vf + t0 * DP);
            for (int i = threadIdx.x; i < n_t * DP / 4; i += blockDim.x) tile[i] = src[i];
        }
        __syncthreads();
        if (!active) continue;
#pragma unroll 4
        for (int jj = 0; jj < n_t; ++jj) {
            float s = 0.0f;
#pragma unroll
            for (int g = 0; g < DP / 4; ++g) {
                const float4 b = tile[jj * (DP / 4) + g];
                const float d0 = xq[4 * g] - b.x, d1 = xq[4 * g + 1] - b.y, d2 = xq[4 * g + 2] - b.z,
                            d3 = xq[4 * g + 3] - b.w;
                s = fmaf(d0, d0, s); s = fmaf(d1, d1, s); s = fmaf(d2, d2, s); s = fmaf(d3, d3, s);
            }
            if (s <= thr32) {  // survivor: exact FP64 recheck (K4)
                const int64_t j = t0 + jj;
                if (j != q) {
                    const double s64 = exact_sq<D>(V + q * D, V + j * D);
                    if (s64 <= r2) {
                        if (FILL) { rowval[pos] = j + 1; nzval[pos] = sqrt(s64); ++pos; }
                        if (MODE == 2 && cnt < cap) {
                            slab_j[w * cap + cnt] = (int)j;
                            slab_s[w * cap + cnt] = s64;
                        }
                        ++cnt;
                    }
                }
            }
        }
    }
    if (!FILL && active) counts[w] = cnt;
}

// slab -> CSC: one warp per column, coalesced reads of the slab row, contiguous Int64/Float64 bursts
__global__ void __launch_bounds__(256)
slab_to_csc(const int *__restrict__ slab_j, const double *__restrict__ slab_s, int cap, int64_t nq,
            const int64_t *__restrict__ colptr, int64_t *__restrict__ rowval, double *__restrict__ nzval) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t w = gw; w < nq; w += nw) {
        const int64_t base = colptr[w] - 1;
        const int k = (int)(colptr[w + 1] - colptr[w]);
        for (int e = lane; e < k; e += 32) {
            rowval[base + e] = (int64_t)slab_j[w * cap + e] + 1;
            nzval[base + e] = sqrt(slab_s[w * cap + e]);
        }
    }
}
// slab -> CSC after the symmetric tensor-core sweep.  A slab row holds the column's entries with a larger index than
// the column at the front (appended by the column's own thread: already ascending) and those with a smaller index at
// the back (appended by their own rows' threads through an atomic slot: unordered).  One block per column sorts the
// back part by sample index in shared memory (bitonic on index << 32 | slot, squared distances parked by slot) and
// writes  sorted(back) ++ front.  np = power of two >= every column's back part, 16 bytes of shared memory each.
// KeyT = uint32_t when (bits of N) + log2(np) <= 32 (key = index << log2(np) | slot), else uint64_t (index << 32 | slot).
// A compare-exchange stage with stride <= 32 only touches the 64-element segment of the pairs a warp owns (pair p
// belongs to segment p >> 5, and a warp always takes whole segments), so those stages synchronise the warp, not the
// block: for 256 keys 6 of the 36 stages need __syncthreads.
template <class KeyT>
__global__ void __launch_bounds__(128)
slab_merge_to_csc(const int *__restrict__ slab_j, const double *__restrict__ slab_s, int cap, int np, int slot_bits, int min_kr,
                  int64_t nq, const int *__restrict__ own, const int *__restrict__ remote, const int64_t *__restrict__ colptr,
                  int64_t *__restrict__ rowval, double *__restrict__ nzval) {
    extern __shared__ unsigned long long s_sort[];  // np squared distances, then np keys
    double *sv = reinterpret_cast<double *>(s_sort);
    KeyT *key = reinterpret_cast<KeyT *>(s_sort + np);
    const KeyT slot_mask = (KeyT)((KeyT(1) << slot_bits) - 1);
    for (int64_t w = blockIdx.x; w < nq; w += gridDim.x) {
        const int64_t base = colptr[w] - 1;
        const int kr = remote[w], ko = own[w];
        if (kr <= min_kr) continue;  // block-uniform: handled by slab_merge_warp
        int n = 64;
        while (n < kr) n <<= 1;  // block-uniform: the smallest power of two that holds the unordered part
        for (int e = threadIdx.x; e < n; e += blockDim.x) {
            if (e < kr) {
                const size_t at = (size_t)w * cap + (cap - 1 - e);
                key[e] = (KeyT)(((KeyT)(unsigned)slab_j[at] << slot_bits) | (KeyT)e);
                sv[e] = slab_s[at];
            } else {
                key[e] = (KeyT)~KeyT(0);
            }
        }
        __syncthreads();
        for (int size = 2; size <= n; size <<= 1)
            for (int stride = size >> 1; stride > 0; stride >>= 1) {
                for (int t = threadIdx.x; t < n / 2; t += blockDim.x) {
                    const int lo = ((t & ~(stride - 1)) << 1) | (t & (stride - 1)), hi = lo | stride;
                    const bool up = (lo & size) == 0;
                    const KeyT a = key[lo], b = key[hi];
                    if ((a > b) == up) { key[lo] = b; key[hi] = a; }
                }
                const int next = stride > 1 ? (stride >> 1) : size;  // stride of the stage that follows
                if (stride >= 64 || next >= 64) __syncthreads(); else __syncwarp();
            }
        __syncthreads();
        for (int e = threadIdx.x; e < kr; e += blockDim.x) {
            const KeyT ky = key[e];
            rowval[base + e] = (int64_t)(ky >> slot_bits) + 1;
            nzval[base + e] = sqrt(sv[(unsigned)(ky & slot_mask)]);
        }
        for (int e = threadIdx.x; e < ko; e += blockDim.x) {
            rowval[base + kr + e] = (int64_t)slab_j[(size_t)w * cap + e] + 1;
            nzval[base + kr + e] = sqrt(slab_s[(size_t)w * cap + e]);
        }
        __syncthreads();
    }
}
// The same conversion with one WARP per column and the keys in registers (K per lane, element e = 32 r + lane):
// compare-exchange stages with a stride below 32 are one shuffle per key, the others are register-to-register, and
// nothing synchronises a block.  Key = index << 10 | slot (needs N < 2^22 and at most 1024 unordered entries; other
// columns are left to slab_merge_to_csc).  After the sort every lane knows (index, slot) of its output positions and
// fetches the squared distance from the slab row by slot.
template <int K>
__device__ __forceinline__ void warp_bitonic(unsigned (&k)[K], int lane) {
#pragma unroll
    for (int size = 2; size <= 32 * K; size <<= 1) {
#pragma unroll
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            if (stride >= 32) {
                const int rs = stride >> 5;
#pragma unroll
                for (int r = 0; r < K; ++r) {
                    if ((r & rs) == 0) {
                        const bool up = ((r << 5) & size) == 0;   // size >= 64 here: the bit lives in r
                        const unsigned a = k[r], b = k[r | rs];
                        const unsigned lo = min(a, b), hi = max(a, b);
                        k[r] = up ? lo : hi;
                        k[r | rs] = up ? hi : lo;
                    }
                }
            } else {
                const bool lower = (lane & stride) == 0;
#pragma unroll
                for (int r = 0; r < K; ++r) {
                    const unsigned o = __shfl_xor_sync(0xffffffffu, k[r], stride);
                    const bool up = (((r << 5) | lane) & size) == 0;
                    k[r] = (lower == up) ? min(k[r], o) : max(k[r], o);
                }
            }
        }
    }
}
template <int K>
__device__ __forceinline__ void merge_column_warp(const int *__restrict__ sj, const double *__restrict__ ss, int cap, int kr,
                                                  int64_t *__restrict__ rv, double *__restrict__ nz, int lane) {
    unsigned k[K];
#pragma unroll
    for (int r = 0; r < K; ++r) {
        const int e = (r << 5) | lane;
        k[r] = e < kr ? (((unsigned)sj[cap - 1 - e] << 10) | (unsigned)e) : 0xffffffffu;
    }
    warp_bitonic<K>(k, lane);
#pragma unroll
    for (int r = 0; r < K; ++r) {
        const int e = (r << 5) | lane;
        if (e < kr) {
            rv[e] = (int64_t)(k[r] >> 10) + 1;
            nz[e] = sqrt(ss[cap - 1 - (int)(k[r] & 1023u)]);
        }
    }
}
// WIDE = false: columns with at most 512 unordered entries; WIDE = true: those with 513 .. 1024 (32 keys per lane:
// a kernel of its own so that the common case does not pay for its registers)
template <bool WIDE>
__global__ void __launch_bounds__(128)
slab_merge_warp(const int *__restrict__ slab_j, const double *__restrict__ slab_s, int cap, int64_t nq,
                const int *__restrict__ own, const int *__restrict__ remote, const int64_t *__restrict__ colptr,
                int64_t *__restrict__ rowval, double *__restrict__ nzval) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t w = gw; w < nq; w += nw) {
        const int kr = remote[w], ko = own[w];
        if (WIDE ? (kr <= 512 || kr > 1024) : (kr > 512)) continue;  // more than 1024: the block-per-column kernel
        const int64_t base = colptr[w] - 1;
        const int *sj = slab_j + (size_t)w * cap;
        const double *ss = slab_s + (size_t)w * cap;
        int64_t *rv = rowval + base;
        double *nz = nzval + base;
        if (WIDE) merge_column_warp<32>(sj, ss, cap, kr, rv, nz, lane);
        else if (kr > 256) merge_column_warp<16>(sj, ss, cap, kr, rv, nz, lane);
        else if (kr > 128) merge_column_warp<8>(sj, ss, cap, kr, rv, nz, lane);
        else if (kr > 64) merge_column_warp<4>(sj, ss, cap, kr, rv, nz, lane);
        else if (kr > 0) merge_column_warp<2>(sj, ss, cap, kr, rv, nz, lane);
        for (int e = lane; e < ko; e += 32) {   // the column's own entries: already ascending
            rv[kr + e] = (int64_t)sj[e] + 1;
            nz[kr + e] = sqrt(ss[e]);
        }
    }
}
__global__ void add_counts(const int *__restrict__ a, const int *__restrict__ b, int64_t n, int *__restrict__ out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = a[i] + b[i];
}
__global__ void max_count(const int *__restrict__ counts, int64_t n, int *__restrict__ out) {
    int m = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) m = max(m, counts[i]);
    for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

// threshold for the FP32 pass: every pair with exact s <= r^2 satisfies s32 <= thr (see DESIGN.md)
static float prefilter_threshold(double r, int D, double M) {
    const double u = 5.9604644775390625e-08;  // 2^-24
    const double e = 2.0 * u * M * (1.0 + u);
    double thr = r * r + 2.0 * (2.0 * e * sqrt((double)D) * r + 2.0 * u * r * r + D * (e + u * r) * (e + u * r));
    thr *= 1.0 + (D + 4) * 2.0 * u;
    float f = (float)thr;
    while ((double)f < thr) f = nextafterf(f, INFINITY);
    return nextafterf(f, INFINITY);
}

template <int D>
static int brute_build(mpb200_samples *s, double r, mpb200_table *t) {
    constexpr int DP = (D + 3) & ~3;
    Context &c = ctx();
    cudaStream_t st = c.stream;
    const int64_t N = s->N, nq = s->q1 - s->q0;
    const double *V = s->V.as<double>();
    const double *bb = s->h_bbox;
    double M = 0;
    for (int i = 0; i < 2 * D; ++i) M = fmax(M, fabs(bb[i]));
    const float thr32 = prefilter_threshold(r, D, M);
    if (!(M < 1e18)) return fail(MPB200_EARG, "sample coordinates out of range for the FP32 prefilter");

    // tensor-core prefilter (tc_rball.cu) for 4 <= d <= 14; MPB200_NO_TC=1 selects the FP32 CUDA-core sweep
    static const bool no_tc = getenv("MPB200_NO_TC") != nullptr;
    constexpr bool kTcDim = (D >= 4 && D <= 14);
    // ... and it is used only while its error band stays tight (DESIGN.md 10): otherwise the CUDA-core form
    const bool use_tc = kTcDim && !no_tc && tc_band_is_tight(s, r);
    TcPlan plan = {nullptr, nullptr, 0, 0.0f};
    phase_bank(MPB200_OP_TABLE);
    phase_mark(0);
    float *Vf = nullptr;
    if (use_tc) {
        if constexpr (kTcDim) {
            if (int rc = tc_prepare_operands<D>(s, r, &plan)) return rc;
        }
    } else {
        if (int rc = s->sorted_pos.reserve(sizeof(float) * (size_t)(N * DP + 4))) return rc;  // reused as the FP32 copy
        Vf = s->sorted_pos.as<float>();
        to_float_padded<D><<<(unsigned)ceil_div(N, 256), 256, 0, st>>>(V, N, Vf);
        MPB_LAUNCHED();
    }
    if (int rc = t->counts.reserve(sizeof(int) * (size_t)(3 * nq + 4))) return rc;  // totals | own | partner appends
    if (int rc = t->colptr.reserve(sizeof(int64_t) * (size_t)(nq + 1))) return rc;
    const unsigned nb = (unsigned)ceil_div(nq > 0 ? nq : 1, kBrThreads);
    const double r2 = r * r;
    int *counts = t->counts.as<int>();
    int *d_max = reinterpret_cast<int *>(c.d_scalar + 2);
    phase_mark(1);
    // ---- slab capacity from a probe of up to 2048 query columns (exact counts for those columns)
    int cap = 0;
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    if (nq > 0) {
        const int64_t probe = nq < 2048 ? nq : 2048;
        MPB_CUDA(cudaMemsetAsync(d_max, 0, sizeof(int), st));
        if (use_tc) {
            if constexpr (kTcDim) {
                if (int rc = tc_sweep<D>(s, plan, r, probe, counts, 0, nullptr, nullptr)) return rc;
            }
        } else {
            brute_rball_kernel<D, 0><<<(unsigned)ceil_div(probe, kBrThreads), kBrThreads, 0, st>>>(
                V, Vf, N, s->q0, probe, r2, thr32, counts, nullptr, nullptr, nullptr, 0, nullptr, nullptr);
            MPB_LAUNCHED();
        }
        max_count<<<8, 256, 0, st>>>(counts, probe, d_max);
        MPB_LAUNCHED();
        int h_max = 0;
        MPB_CUDA(cudaMemcpyAsync(&h_max, d_max, sizeof(int), cudaMemcpyDeviceToHost, st));
        MPB_CUDA(cudaStreamSynchronize(st));
        cap = (probe == nq) ? h_max : (h_max + h_max / 2 + 64);
        cap = (cap + 31) & ~31;
        // slabs must leave room for the table itself; otherwise use the two-sweep path
        // ... counting what a rebuild can reuse: the table's own buffers and the blocks parked in the cache
        const double need = 12.0 * (double)cap * (double)nq + 16.0 * 0.8 * (double)cap * (double)nq;
        const double avail = (double)free_b + (double)cache_parked_bytes() + (double)t->scratch.cap +
                             (double)t->rowval.cap + (double)t->nzval.cap;
        if (cap == 0 || need > 0.8 * avail) cap = 0;
    }
    bool single = cap > 0;
    // full-range tensor-core builds multiply every unordered pair once and append it to both columns (tc_rball.cu,
    // MODE 3); MPB200_TC_FULL=1 keeps the one-sided sweep.  The sorting conversion holds a column in shared memory.
    static const bool tc_full = getenv("MPB200_TC_FULL") != nullptr;
    const bool symmetric = single && use_tc && !tc_full && nq == N && s->q0 == 0 && cap <= 8192;  // 8192 entries = 128 KB of shared memory
    if (single) {
        if (int rc = t->scratch.reserve(12 * (size_t)cap * (size_t)nq + 64)) return rc;
        double *slab_s = t->scratch.as<double>();
        int *slab_j = reinterpret_cast<int *>(slab_s + (size_t)cap * (size_t)nq);
        if (use_tc) {
            if constexpr (kTcDim) {
                if (symmetric) {
                    int *own = counts + nq + 2, *remote = own + nq;
                    if (int rc = tc_sweep<D>(s, plan, r, nq, own, cap, slab_j, slab_s, remote)) return rc;
                    add_counts<<<(unsigned)(ctx().sm_count * 4), 256, 0, st>>>(own, remote, nq, counts);
                    MPB_LAUNCHED();
                } else {
                    if (int rc = tc_sweep<D>(s, plan, r, nq, counts, cap, slab_j, slab_s)) return rc;
                }
            }
        } else {
            brute_rball_kernel<D, 2><<<nb, kBrThreads, 0, st>>>(V, Vf, N, s->q0, nq, r2, thr32, counts, nullptr, nullptr,
                                                               nullptr, cap, slab_j, slab_s);
            MPB_LAUNCHED();
        }
        MPB_CUDA(cudaMemsetAsync(d_max, 0, sizeof(int), st));
        max_count<<<64, 256, 0, st>>>(counts, nq, d_max);
        MPB_LAUNCHED();
    } else if (nq > 0) {
        if (use_tc) {
            if constexpr (kTcDim) {
                if (int rc = tc_sweep<D>(s, plan, r, nq, counts, 0, nullptr, nullptr)) return rc;
            }
        } else {
            brute_rball_kernel<D, 0><<<nb, kBrThreads, 0, st>>>(V, Vf, N, s->q0, nq, r2, thr32, counts, nullptr, nullptr,
                                                               nullptr, 0, nullptr, nullptr);
            MPB_LAUNCHED();
        }
    }
    if (int rc = exclusive_scan<int, int64_t>(counts, nq, t->colptr.as<int64_t>(), (int64_t)1, s->scan_tmp, c.d_scalar))
        return rc;
    phase_mark(2);
    MPB_CUDA(cudaMemcpyAsync(c.h_scalar, c.d_scalar, sizeof(int64_t) * 3, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    const int64_t nnz = c.h_scalar[0];
    if (single && *reinterpret_cast<int *>(c.h_scalar + 2) > cap) single = false;  // a slab overflowed: two-sweep fill
    if (int rc = t->rowval.reserve(sizeof(int64_t) * (size_t)(nnz + 1))) return rc;
    if (int rc = t->nzval.reserve(sizeof(double) * (size_t)(nnz + 1))) return rc;
    phase_mark(3);
    if (nq > 0 && nnz > 0) {
        bool counted = false;
        if (single) {
            const double *slab_s = t->scratch.as<double>();
            const int *slab_j = reinterpret_cast<const int *>(slab_s + (size_t)cap * (size_t)nq);
            if (symmetric) {
                int np = 64, slot_bits = 6;
                while (np < cap) { np <<= 1; ++slot_bits; }
                int idx_bits = 1;
                while ((int64_t(1) << idx_bits) < N) ++idx_bits;
                static const bool block_only = getenv("MPB200_SLAB_BLOCK_SORT") != nullptr;
                const bool warp_sort = idx_bits <= 22 && !block_only;   // key = index << 10 | slot in 32 bits
                if (warp_sort) {
                    slab_merge_warp<false><<<(unsigned)(ctx().sm_count * 16), 128, 0, st>>>(
                        slab_j, slab_s, cap, nq, counts + nq + 2, counts + 2 * nq + 2, t->colptr.as<int64_t>(),
                        t->rowval.as<int64_t>(), t->nzval.as<double>());
                    MPB_LAUNCHED();
                    if (cap > 512) {
                        slab_merge_warp<true><<<(unsigned)(ctx().sm_count * 8), 128, 0, st>>>(
                            slab_j, slab_s, cap, nq, counts + nq + 2, counts + 2 * nq + 2, t->colptr.as<int64_t>(),
                            t->rowval.as<int64_t>(), t->nzval.as<double>());
                        MPB_LAUNCHED();
                    }
                }
                if (!warp_sort || cap > 1024) {   // every column, or only those with more than 1024 unordered entries
                    const int min_kr = warp_sort ? 1024 : -1;
                    const bool narrow = idx_bits + slot_bits <= 32;
                    const size_t smem = (narrow ? 12 : 16) * (size_t)np;
                    const unsigned gs = (unsigned)std::min<int64_t>(nq, (int64_t)ctx().sm_count * 32);
                    if (narrow) {
                        MPB_CUDA(cudaFuncSetAttribute(slab_merge_to_csc<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                        slab_merge_to_csc<uint32_t><<<gs, 128, smem, st>>>(slab_j, slab_s, cap, np, slot_bits, min_kr, nq, counts + nq + 2,
                                                                           counts + 2 * nq + 2, t->colptr.as<int64_t>(),
                                                                           t->rowval.as<int64_t>(), t->nzval.as<double>());
                    } else {
                        MPB_CUDA(cudaFuncSetAttribute(slab_merge_to_csc<uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                        slab_merge_to_csc<uint64_t><<<gs, 128, smem, st>>>(slab_j, slab_s, cap, np, 32, min_kr, nq, counts + nq + 2,
                                                                           counts + 2 * nq + 2, t->colptr.as<int64_t>(),
                                                                           t->rowval.as<int64_t>(), t->nzval.as<double>());
                    }
                } else {
                    counted = true;   // the warp kernel was the only launch and has been counted
                }
            } else
            slab_to_csc<<<(unsigned)(ctx().sm_count * 8), 256, 0, st>>>(slab_j, slab_s, cap, nq, t->colptr.as<int64_t>(),
                                                                       t->rowval.as<int64_t>(), t->nzval.as<double>());
        } else {
            if (!Vf) {  // two-sweep fill after a tensor-core count: the FP32 copy is built now (aux holds it)
                if (int rc = s->q_order.reserve(sizeof(float) * (size_t)(N * DP + 4))) return rc;
                Vf = s->q_order.as<float>();
                to_float_padded<D><<<(unsigned)ceil_div(N, 256), 256, 0, st>>>(V, N, Vf);
                MPB_LAUNCHED();
            }
            brute_rball_kernel<D, 1><<<nb, kBrThreads, 0, st>>>(V, Vf, N, s->q0, nq, r2, thr32, nullptr,
                                                               t->colptr.as<int64_t>(), t->rowval.as<int64_t>(),
                                                               t->nzval.as<double>(), 0, nullptr, nullptr);
        }
        if (!counted) MPB_LAUNCHED();
    }
    phase_mark(4);
    MPB_CUDA(cudaStreamSynchronize(st));
    phases_collect(4);
    t->ncols = nq;
    t->col0 = s->q0;
    t->nnz = nnz;
    t->r = r;
    t->euclid = true;
    t->has_order = false;
    return 0;
}

int brute_inball_build(mpb200_samples *s, double r, mpb200_table *t) {
    s->pt_order_valid = false;  // sorted_pos and q_order are reused as FP32 scratch here
    switch (s->d) {
    case 4: return brute_build<4>(s, r, t);
    case 5: return brute_build<5>(s, r, t);
    case 6: return brute_build<6>(s, r, t);
    case 7: return brute_build<7>(s, r, t);
    case 8: return brute_build<8>(s, r, t);
    case 9: return brute_build<9>(s, r, t);
    case 10: return brute_build<10>(s, r, t);
    case 11: return brute_build<11>(s, r, t);
    case 12: return brute_build<12>(s, r, t);
    case 13: return brute_build<13>(s, r, t);
    case 14: return brute_build<14>(s, r, t);
    case 15: return brute_build<15>(s, r, t);
    case 16: return brute_build<16>(s, r, t);
    case 1: return brute_build<1>(s, r, t);
    default: return fail(MPB200_EARG, "all-pairs r-ball supports d = 1 and 4..16 (got %d)", s->d);
    }
}

}  // namespace mpb
