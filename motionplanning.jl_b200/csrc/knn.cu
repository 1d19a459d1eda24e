// knn.cu -- k-nearest connections on top of the neighbour tables.
//
// The reference exports knn / knnF / knnB / mutualknn* (nearneighbors.jl:9-11) and FMT*'s connections = :K branch
// calls mutualknnF! / knnB! (fmt.jl:6,17-19,70,72) -- but none of them is defined anywhere in the reference
// (SURVEY quirk Q6: `:K` throws).  PARITY UNPINNED; the specification implemented here, and restated in
// oracle/oracle.py (knn_brute / mutual_knn):
//   knn(v, k)        = the k samples j != v with the smallest stored value (distance / steering cost), ties broken
//                      towards the smaller index; returned like every neighbourhood: ascending indices + values;
//   mutualknnF(v, k) = knnF(v, k)  union  { w : v in knnB(w, k) }   (values cost(v -> w) from either side).
// Both are TABLE operations, metric-agnostic: mpb200_table_knn keeps the k best entries of every column of an
// r-ball table that holds at least k entries per column (the caller grows r until it does), and
// mpb200_table_union_transpose forms  A[:, v]  union  { w : v in B[:, w] }.
// One block per column; a column lives in shared memory (bitonic networks on packed keys).
#include "common.cuh"
#include "scan.cuh"
#include <algorithm>
#include <new>

namespace mpb {

constexpr int kKnnThreads = 128;

// ascending bitonic sort of n (power of two) 64-bit keys in shared memory, whole block
__device__ __forceinline__ void block_bitonic(unsigned long long *key, int n) {
    for (int size = 2; size <= n; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = threadIdx.x; t < n / 2; t += blockDim.x) {
                const int lo = ((t & ~(stride - 1)) << 1) | (t & (stride - 1)), hi = lo | stride;
                const bool up = (lo & size) == 0;
                const unsigned long long a = key[lo], b = key[hi];
                if ((a > b) == up) { key[lo] = b; key[hi] = a; }
            }
            __syncthreads();
        }
}
__device__ __forceinline__ int pow2_at_least(int k) {
    int n = 32;
    while (n < k) n <<= 1;
    return n;
}

__global__ void knn_lengths(const int64_t *__restrict__ colptr, int64_t ncols, int k, int *__restrict__ cnt,
                            unsigned long long *__restrict__ n_short) {
    unsigned long long mine = 0;
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < ncols; w += (int64_t)gridDim.x * blockDim.x) {
        const int len = (int)(colptr[w + 1] - colptr[w]);
        cnt[w] = len < k ? len : k;
        mine += len < k ? 1 : 0;
    }
    if (mine) atomicAdd(n_short, mine);
}

// ascending bitonic sort of n (power of two) (value, slot) pairs, lexicographic, whole block
__device__ __forceinline__ void block_bitonic2(unsigned long long *val, unsigned *slot, int n) {
    for (int size = 2; size <= n; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = threadIdx.x; t < n / 2; t += blockDim.x) {
                const int lo = ((t & ~(stride - 1)) << 1) | (t & (stride - 1)), hi = lo | stride;
                const bool up = (lo & size) == 0;
                const unsigned long long va = val[lo], vb = val[hi];
                const unsigned sa = slot[lo], sb = slot[hi];
                const bool gt = (va > vb) || (va == vb && sa > sb);
                if (gt == up) { val[lo] = vb; val[hi] = va; slot[lo] = sb; slot[hi] = sa; }
            }
            __syncthreads();
        }
}

// keep the k entries with the smallest (value, row) of every column; rows stay ascending.
// shared memory: np 64-bit values + np 32-bit slots
__global__ void __launch_bounds__(kKnnThreads)
knn_select_kernel(const int64_t *__restrict__ colptr, const int64_t *__restrict__ rowval, const double *__restrict__ nzval,
                  int64_t ncols, int k, int np, const int64_t *__restrict__ colptr_out, int64_t *__restrict__ rowval_out,
                  double *__restrict__ nzval_out) {
    extern __shared__ unsigned long long s_key[];
    unsigned *s_slot = reinterpret_cast<unsigned *>(s_key + np);
    for (int64_t w = blockIdx.x; w < ncols; w += gridDim.x) {
        const int64_t base = colptr[w] - 1, obase = colptr_out[w] - 1;
        const int len = (int)(colptr[w + 1] - colptr[w]);
        if (len <= k) {  // short column: kept whole (block-uniform branch)
            for (int e = threadIdx.x; e < len; e += blockDim.x) {
                rowval_out[obase + e] = rowval[base + e];
                nzval_out[obase + e] = nzval[base + e];
            }
            continue;
        }
        // pass 1: order by (value, slot).  Stored values are non-negative doubles, so their bit patterns order like
        // the numbers; the slot is the position in the column = ascending row index: equal values keep the smaller index.
        const int n = pow2_at_least(len);
        for (int e = threadIdx.x; e < n; e += blockDim.x) {
            s_key[e] = e < len ? (unsigned long long)__double_as_longlong(nzval[base + e]) : ~0ULL;
            s_slot[e] = (unsigned)e;
        }
        __syncthreads();
        block_bitonic2(s_key, s_slot, n);
        // pass 2: the k winners back into slot (= row) order
        const int n2 = pow2_at_least(k);
        for (int e = threadIdx.x; e < n2; e += blockDim.x) s_key[e] = e < k ? (unsigned long long)s_slot[e] : ~0ULL;
        __syncthreads();
        block_bitonic(s_key, n2);
        for (int e = threadIdx.x; e < k; e += blockDim.x) {
            const int slot = (int)s_key[e];
            rowval_out[obase + e] = rowval[base + slot];
            nzval_out[obase + e] = nzval[base + slot];
        }
        __syncthreads();
    }
}

// ---- transpose of B: per-row counts, scatter (unordered inside a row) ------------------------------------------
__global__ void count_rows_kernel(const int64_t *__restrict__ rowval, int64_t nnz, int *__restrict__ cnt) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (int64_t)gridDim.x * blockDim.x)
        atomicAdd(&cnt[rowval[e] - 1], 1);
}
__global__ void __launch_bounds__(256)
scatter_rows_kernel(const int64_t *__restrict__ colptr, const int64_t *__restrict__ rowval, const double *__restrict__ nzval,
                    int64_t ncols, int64_t col0, const int64_t *__restrict__ ptrT, int *__restrict__ cursor,
                    int *__restrict__ rowT, double *__restrict__ valT) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t w = gw; w < ncols; w += nw)
        for (int64_t e = colptr[w] - 1 + lane; e < colptr[w + 1] - 1; e += 32) {
            const int64_t v = rowval[e] - 1;
            const int64_t at = ptrT[v] - 1 + atomicAdd(&cursor[v], 1);
            rowT[at] = (int)(col0 + w);
            valT[at] = nzval[e];
        }
}

// out[:, v] = a[:, v]  union  T[v]; FILL = false: lengths only.  Keys = row << 14 | source bit << 13 | slot.
template <bool FILL>
__global__ void __launch_bounds__(kKnnThreads)
union_kernel(const int64_t *__restrict__ a_colptr, const int64_t *__restrict__ a_row, const double *__restrict__ a_val,
             const int64_t *__restrict__ ptrT, const int *__restrict__ rowT, const double *__restrict__ valT,
             int64_t ncols, int np, int *__restrict__ cnt, const int64_t *__restrict__ colptr_out,
             int64_t *__restrict__ rowval_out, double *__restrict__ nzval_out) {
    extern __shared__ unsigned long long s_key[];
    (void)np;
    __shared__ int s_part[kKnnThreads + 1];
    for (int64_t v = blockIdx.x; v < ncols; v += gridDim.x) {
        const int64_t ab = a_colptr[v] - 1, tb = ptrT[v] - 1;
        const int la = (int)(a_colptr[v + 1] - a_colptr[v]), lt = (int)(ptrT[v + 1] - ptrT[v]);
        const int len = la + lt, n = pow2_at_least(len);
        for (int e = threadIdx.x; e < n; e += blockDim.x) {
            unsigned long long ky = ~0ULL;
            if (e < la) ky = ((unsigned long long)(a_row[ab + e] - 1) << 14) | (unsigned)e;
            else if (e < len) ky = ((unsigned long long)(unsigned)rowT[tb + e - la] << 14) | (1ULL << 13) | (unsigned)(e - la);
            s_key[e] = ky;
        }
        __syncthreads();
        block_bitonic(s_key, n);
        // keep the first element of every run of equal rows (a's copy sorts before T's)
        const int per = (n + kKnnThreads - 1) / kKnnThreads, e0 = threadIdx.x * per;
        int local = 0;
        for (int e = e0; e < e0 + per && e < len; ++e)
            local += (e == 0 || (s_key[e] >> 14) != (s_key[e - 1] >> 14)) ? 1 : 0;
        s_part[threadIdx.x + 1] = local;
        if (threadIdx.x == 0) s_part[0] = 0;
        __syncthreads();
        if (threadIdx.x == 0)
            for (int i = 1; i <= kKnnThreads; ++i) s_part[i] += s_part[i - 1];
        __syncthreads();
        if (!FILL) {
            if (threadIdx.x == 0) cnt[v] = s_part[kKnnThreads];
        } else {
            const int64_t ob = colptr_out[v] - 1;
            int pos = s_part[threadIdx.x];
            for (int e = e0; e < e0 + per && e < len; ++e) {
                const unsigned long long ky = s_key[e];
                if (e == 0 || (ky >> 14) != (s_key[e - 1] >> 14)) {
                    const int slot = (int)(ky & 0x1fffULL);
                    rowval_out[ob + pos] = (int64_t)(ky >> 14) + 1;
                    nzval_out[ob + pos] = ((ky >> 13) & 1ULL) ? valT[tb + slot] : a_val[ab + slot];
                    ++pos;
                }
            }
        }
        __syncthreads();
    }
}

__global__ void max_len_kernel(const int64_t *__restrict__ p1, const int64_t *__restrict__ p2, int64_t n, int *__restrict__ out) {
    int m = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int l = (int)(p1[i + 1] - p1[i]);
        if (p2) l += (int)(p2[i + 1] - p2[i]);
        m = max(m, l);
    }
    for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

static int copy_meta(const mpb200_table *src, mpb200_table *dst) {
    dst->ncols = src->ncols; dst->col0 = src->col0; dst->r = src->r; dst->euclid = src->euclid;
    dst->src_N = src->src_N; dst->src_d = src->src_d; dst->src_serial = src->src_serial; dst->edge_bits_valid = false; dst->has_order = false;
    if (src->has_order && src->ncols > 0) {  // same columns: the cell-order visiting list stays valid
        if (int rc = dst->col_order.reserve(sizeof(int) * (size_t)(src->ncols + 1))) return rc;
        MPB_CUDA(cudaMemcpyAsync(dst->col_order.p, src->col_order.p, sizeof(int) * (size_t)src->ncols, cudaMemcpyDeviceToDevice, ctx().stream));
        dst->has_order = true;
    }
    return 0;
}

__global__ void short_columns_kernel(const int64_t *__restrict__ colptr, int64_t ncols, int k, unsigned long long *__restrict__ n_short) {
    unsigned long long mine = 0;
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < ncols; w += (int64_t)gridDim.x * blockDim.x)
        mine += (colptr[w + 1] - colptr[w]) < k ? 1 : 0;
    for (int o = 16; o; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(n_short, mine);
}

// columns of t with fewer than k entries (the cheap question "is the radius large enough?" before any selection)
int table_short_columns_device(const mpb200_table *t, int k, int64_t *short_cols) {
    Context &c = ctx();
    cudaStream_t st = c.stream;
    MPB_CUDA(cudaMemsetAsync(c.d_scalar + 3, 0, sizeof(int64_t), st));
    if (t->ncols > 0) {
        const unsigned g = (unsigned)std::min<int64_t>(std::max<int64_t>(ceil_div(t->ncols, 256), 1), (int64_t)c.sm_count * 8);
        short_columns_kernel<<<g, 256, 0, st>>>(t->colptr.as<int64_t>(), t->ncols, k, reinterpret_cast<unsigned long long *>(c.d_scalar + 3));
        MPB_LAUNCHED();
    }
    MPB_CUDA(cudaMemcpyAsync(c.h_scalar + 3, c.d_scalar + 3, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    *short_cols = c.h_scalar[3];
    return 0;
}

int table_knn_device(const mpb200_table *t, int k, mpb200_table *out, int64_t *short_cols, DevBuf &scan_tmp) {
    Context &c = ctx();
    cudaStream_t st = c.stream;
    const int64_t nc = t->ncols;
    if (int rc = out->counts.reserve(sizeof(int) * (size_t)(nc + 2))) return rc;
    if (int rc = out->colptr.reserve(sizeof(int64_t) * (size_t)(nc + 1))) return rc;
    int *d_max = reinterpret_cast<int *>(c.d_scalar + 2);
    unsigned long long *d_short = reinterpret_cast<unsigned long long *>(c.d_scalar + 3);
    MPB_CUDA(cudaMemsetAsync(c.d_scalar + 2, 0, sizeof(int64_t) * 2, st));
    const unsigned g = (unsigned)std::min<int64_t>(std::max<int64_t>(ceil_div(nc, 256), 1), (int64_t)c.sm_count * 8);
    if (nc > 0) {
        knn_lengths<<<g, 256, 0, st>>>(t->colptr.as<int64_t>(), nc, k, out->counts.as<int>(), d_short);
        MPB_LAUNCHED();
        max_len_kernel<<<g, 256, 0, st>>>(t->colptr.as<int64_t>(), nullptr, nc, d_max);
        MPB_LAUNCHED();
    }
    if (int rc = exclusive_scan<int, int64_t>(out->counts.as<int>(), nc, out->colptr.as<int64_t>(), (int64_t)1, scan_tmp, c.d_scalar))
        return rc;
    MPB_CUDA(cudaMemcpyAsync(c.h_scalar, c.d_scalar, sizeof(int64_t) * 4, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    const int64_t nnz = c.h_scalar[0];
    const int max_len = *reinterpret_cast<int *>(c.h_scalar + 2);
    *short_cols = c.h_scalar[3];
    if (max_len > 8192) return fail(MPB200_EARG, "k-nearest selection holds a column in shared memory: at most 8192 entries per column (got %d); use a smaller radius", max_len);
    if (int rc = out->rowval.reserve(sizeof(int64_t) * (size_t)(nnz + 1))) return rc;
    if (int rc = out->nzval.reserve(sizeof(double) * (size_t)(nnz + 1))) return rc;
    if (nc > 0 && nnz > 0) {
        int np = 32;
        while (np < max_len) np <<= 1;
        const size_t smem = 12 * (size_t)np;
        MPB_CUDA(cudaFuncSetAttribute(knn_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const unsigned gs = (unsigned)std::min<int64_t>(nc, (int64_t)c.sm_count * 16);
        knn_select_kernel<<<gs, kKnnThreads, smem, st>>>(t->colptr.as<int64_t>(), t->rowval.as<int64_t>(), t->nzval.as<double>(),
                                                         nc, k, np, out->colptr.as<int64_t>(), out->rowval.as<int64_t>(),
                                                         out->nzval.as<double>());
        MPB_LAUNCHED();
    }
    out->nnz = nnz;
    return copy_meta(t, out);
}

int table_union_transpose_device(const mpb200_table *a, const mpb200_table *b, mpb200_table *out, DevBuf &scan_tmp) {
    Context &c = ctx();
    cudaStream_t st = c.stream;
    const int64_t nc = a->ncols;
    // transpose of b: ptrT (int64, nc+1) | cursor / counts (int, nc+1) in out->scratch, rowT / valT after them
    if (int rc = out->counts.reserve(sizeof(int) * (size_t)(2 * nc + 4))) return rc;
    if (int rc = out->colptr.reserve(sizeof(int64_t) * (size_t)(nc + 1))) return rc;
    if (int rc = out->scratch.reserve(sizeof(int64_t) * (size_t)(nc + 2) + 12 * (size_t)(b->nnz + 1) + 64)) return rc;
    int64_t *ptrT = out->scratch.as<int64_t>();
    double *valT = reinterpret_cast<double *>(ptrT + nc + 2);
    int *rowT = reinterpret_cast<int *>(valT + b->nnz + 1);
    int *cntT = out->counts.as<int>(), *cursor = cntT + nc + 2;
    MPB_CUDA(cudaMemsetAsync(cntT, 0, sizeof(int) * (size_t)(2 * nc + 4), st));
    const unsigned g = (unsigned)std::min<int64_t>(std::max<int64_t>(ceil_div(b->nnz, 256), 1), (int64_t)c.sm_count * 8);
    if (b->nnz > 0) {
        count_rows_kernel<<<g, 256, 0, st>>>(b->rowval.as<int64_t>(), b->nnz, cntT);
        MPB_LAUNCHED();
    }
    if (int rc = exclusive_scan<int, int64_t>(cntT, nc, ptrT, (int64_t)1, scan_tmp, c.d_scalar + 1)) return rc;
    if (b->nnz > 0) {
        scatter_rows_kernel<<<(unsigned)(c.sm_count * 8), 256, 0, st>>>(b->colptr.as<int64_t>(), b->rowval.as<int64_t>(),
                                                                       b->nzval.as<double>(), b->ncols, b->col0, ptrT, cursor, rowT, valT);
        MPB_LAUNCHED();
    }
    int *d_max = reinterpret_cast<int *>(c.d_scalar + 2);
    MPB_CUDA(cudaMemsetAsync(c.d_scalar + 2, 0, sizeof(int64_t), st));
    const unsigned gm = (unsigned)std::min<int64_t>(std::max<int64_t>(ceil_div(nc, 256), 1), (int64_t)c.sm_count * 8);
    if (nc > 0) {
        max_len_kernel<<<gm, 256, 0, st>>>(a->colptr.as<int64_t>(), ptrT, nc, d_max);
        MPB_LAUNCHED();
    }
    MPB_CUDA(cudaMemcpyAsync(c.h_scalar + 2, c.d_scalar + 2, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    const int max_len = *reinterpret_cast<int *>(c.h_scalar + 2);
    if (max_len > 8192) return fail(MPB200_EARG, "mutual neighbourhoods hold a column in shared memory: at most 8192 entries (got %d)", max_len);
    int np = 32;
    while (np < max_len) np <<= 1;
    const size_t smem = 8 * (size_t)np;
    MPB_CUDA(cudaFuncSetAttribute(union_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MPB_CUDA(cudaFuncSetAttribute(union_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned gs = (unsigned)std::min<int64_t>(std::max<int64_t>(nc, 1), (int64_t)c.sm_count * 16);
    int *cnt = cursor;  // the scatter is done: reuse as the union lengths
    if (nc > 0) {
        union_kernel<false><<<gs, kKnnThreads, smem, st>>>(a->colptr.as<int64_t>(), a->rowval.as<int64_t>(), a->nzval.as<double>(), ptrT,
                                                           rowT, valT, nc, np, cnt, nullptr, nullptr, nullptr);
        MPB_LAUNCHED();
    }
    if (int rc = exclusive_scan<int, int64_t>(cnt, nc, out->colptr.as<int64_t>(), (int64_t)1, scan_tmp, c.d_scalar)) return rc;
    MPB_CUDA(cudaMemcpyAsync(c.h_scalar, c.d_scalar, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    const int64_t nnz = c.h_scalar[0];
    if (int rc = out->rowval.reserve(sizeof(int64_t) * (size_t)(nnz + 1))) return rc;
    if (int rc = out->nzval.reserve(sizeof(double) * (size_t)(nnz + 1))) return rc;
    if (nc > 0 && nnz > 0) {
        union_kernel<true><<<gs, kKnnThreads, smem, st>>>(a->colptr.as<int64_t>(), a->rowval.as<int64_t>(), a->nzval.as<double>(), ptrT,
                                                          rowT, valT, nc, np, nullptr, out->colptr.as<int64_t>(),
                                                          out->rowval.as<int64_t>(), out->nzval.as<double>());
        MPB_LAUNCHED();
    }
    out->nnz = nnz;
    return copy_meta(a, out);
}

}  // namespace mpb
