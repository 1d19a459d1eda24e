// shortcut.cu -- mpb200_shortcut_paths: the cheapest collision-free route through each path's subdivided waypoints
// (specification in include/mpb200.h and DESIGN.md section 10c).
//
// Three launches per call, whatever the number of paths: the nodes are built on the device from the uploaded states
// (shortcut_nodes_kernel); the visibility pass of collide.cu fills one bit per pair a < b of every path; then one CTA per
// path runs the minimum over b = 1..M-1 in order (shortcut_min_kernel) and writes its output row.
#include "shortcut.cuh"
#include "predicates.cuh"
#include <climits>
#include <cmath>
#include <vector>

namespace mpb {

constexpr int kNodeThreads = 256;
constexpr int kMinThreads = 256;

// Node n of a path: Y[i] for n = i k, else Y[i] + t (Y[i+1] - Y[i]) with t = m / k, one rounding per operation.
// Thread q < npaths also zeroes the segment-test count of path q.
__global__ void __launch_bounds__(kNodeThreads)
shortcut_nodes_kernel(const ShortcutPath *__restrict__ paths, int npaths, int64_t nodes_total, int d, int k,
                      const double *__restrict__ Y, double *__restrict__ nodes, ShortcutResult *__restrict__ results) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < nodes_total; g += stride) {
        if (g < npaths) results[g].checks = 0;
        const int q = shortcut_path_of(paths, npaths, g);
        const int n = (int)(g - paths[q].node0);
        const int i = n / k, m = n - i * k;
        const double *y = Y + (paths[q].y0 + i) * d;
        double *out = nodes + g * d;
        if (m == 0) {
            for (int c = 0; c < d; ++c) out[c] = y[c];
        } else {
            const double t = ddiv((double)m, (double)k);
            for (int c = 0; c < d; ++c) out[c] = dadd(y[c], dmul(t, dsub(y[d + c], y[c])));
        }
    }
}

// (value, index) pairs: the smaller value, ties to the smaller index -- the result does not depend on the reduction order
__device__ __forceinline__ bool shortcut_better(double v, int a, double bv, int ba) {
    return v < bv || (v == bv && a < ba);
}

// One CTA per path.  For b = 1..M-1 in order: the threads take the a < b of row b, and for each visibility bit that is
// set form best[a] + cost(a, b) with the cost recomputed from the nodes; a block-wide argmin on (value, a) gives best[b]
// and pred[b].  Then the output row: the pred chain 0 .. M-1 when best[M-1] is finite, else the input states.
template <int D>
__global__ void __launch_bounds__(kMinThreads)
shortcut_min_kernel(const ShortcutPath *__restrict__ paths, int d_rt, int k, const double *__restrict__ nodes,
                    const uint32_t *__restrict__ bits, double *__restrict__ best, int *__restrict__ pred,
                    double *__restrict__ out, ShortcutResult *__restrict__ results) {
    const int d = D > 0 ? D : d_rt;
    const int q = blockIdx.x;
    const ShortcutPath P = paths[q];
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    const double *nd = nodes + P.node0 * d;
    double *bq = best + P.node0;
    int *pq = pred + P.node0;
    __shared__ double s_v[kMinThreads / 32];
    __shared__ int s_a[kMinThreads / 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) { bq[0] = 0.0; pq[0] = -1; }
    __syncthreads();
    for (int b = 1; b < P.M; ++b) {
        const uint32_t *row = bits + P.bit0 + (int64_t)b * P.words;
        const double *xb = nd + (int64_t)b * d;
        double bv = inf;
        int ba = INT_MAX;
        for (int a = threadIdx.x; a < b; a += kMinThreads) {
            if (!((__ldg(row + (a >> 5)) >> (a & 31)) & 1u)) continue;
            const double *xa = nd + (int64_t)a * d;
            double s = 0.0;  // cost(a, b): index order, one rounding per operation
#pragma unroll
            for (int c = 0; c < (D > 0 ? D : kMaxDim); ++c) {
                if (D == 0 && c >= d) break;
                const double e = dsub(xa[c], xb[c]);
                s = dadd(s, dmul(e, e));
            }
            const double v = dadd(bq[a], __dsqrt_rn(s));
            if (shortcut_better(v, a, bv, ba)) { bv = v; ba = a; }
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oa = __shfl_xor_sync(0xffffffffu, ba, o);
            if (shortcut_better(ov, oa, bv, ba)) { bv = ov; ba = oa; }
        }
        if (lane == 0) { s_v[wid] = bv; s_a[wid] = ba; }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < kMinThreads / 32; ++w)
                if (shortcut_better(s_v[w], s_a[w], bv, ba)) { bv = s_v[w]; ba = s_a[w]; }
            bq[b] = bv;  // +inf when no free a gives a finite value
            pq[b] = bv < inf ? ba : -1;
        }
        __syncthreads();  // best[b] is read by every thread from b + 1 on
    }
    const double cost = bq[P.M - 1];
    double *oq = out + P.node0 * d;
    if (cost < inf) {
        if (threadIdx.x == 0) {
            long long len = 1;
            for (int b = P.M - 1; b != 0; b = pq[b]) ++len;
            long long i = len - 1;
            for (int b = P.M - 1;; b = pq[b], --i) {
                for (int c = 0; c < d; ++c) oq[i * d + c] = nd[(int64_t)b * d + c];
                if (b == 0) break;
            }
            results[q].len = len;
            results[q].cost = cost;
        }
    } else {  // not free: the input path unchanged (node i k is Y[i] bit for bit)
        for (int i = threadIdx.x; i < P.L; i += kMinThreads)
            for (int c = 0; c < d; ++c) oq[(int64_t)i * d + c] = nd[(int64_t)i * k * d + c];
        if (threadIdx.x == 0) {
            results[q].len = P.L;
            results[q].cost = inf;
        }
    }
}

static size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

// the three launches of a call, on the library stream, timed as phase 1 (nodes + visibility) and phase 2 (minimum)
static int shortcut_launch(const ShortcutPath *paths, int npaths, int64_t nodes_total, int d, int k, const double *Y,
                           const mpb200_obstacles *o, const mpb200_space_desc *ss, double *nodes, uint32_t *bits,
                           double *best, int *pred, double *out, ShortcutResult *res) {
    Context &c = ctx();
    cudaStream_t st = c.stream;
    phase_bank(MPB200_OP_PATH);
    phase_mark(0);
    const int64_t blocks = ceil_div(nodes_total, kNodeThreads), cap = (int64_t)c.sm_count * 8;
    shortcut_nodes_kernel<<<(unsigned)(blocks < cap ? blocks : cap), kNodeThreads, 0, st>>>(paths, npaths, nodes_total,
                                                                                           d, k, Y, nodes, res);
    MPB_LAUNCHED();
    if (int rc = shortcut_visibility_device(paths, npaths, nodes_total, nodes, d, o, ss, bits, res)) return rc;
    phase_mark(1);
    const unsigned grid = (unsigned)npaths;
    if (d == 2) shortcut_min_kernel<2><<<grid, kMinThreads, 0, st>>>(paths, d, k, nodes, bits, best, pred, out, res);
    else if (d == 3) shortcut_min_kernel<3><<<grid, kMinThreads, 0, st>>>(paths, d, k, nodes, bits, best, pred, out, res);
    else shortcut_min_kernel<0><<<grid, kMinThreads, 0, st>>>(paths, d, k, nodes, bits, best, pred, out, res);
    MPB_LAUNCHED();
    phase_mark(2);
    phases_collect(2);
    return 0;
}

}  // namespace mpb

using namespace mpb;

extern "C" {

int mpb200_shortcut_paths(const double *states_aos, const int64_t *offsets, int64_t npaths, int d,
                          const mpb200_obstacles *o, const mpb200_space_desc *ss, int32_t subdivisions,
                          double *out_states, int64_t out_cap, int64_t *out_len, double *costs, int64_t *pairs,
                          int64_t *segment_checks) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(npaths >= 1, "at least one path is needed");
    MPB_CHECK_ARG(states_aos && offsets && out_len && costs, "NULL argument");
    MPB_CHECK_ARG(subdivisions >= 1, "subdivisions must be >= 1");
    MPB_CHECK_ARG(out_cap >= 0 && (out_states != nullptr || out_cap == 0), "out_states is NULL with out_cap > 0");
    MPB_CHECK_ARG(offsets[0] == 0, "offsets[0] must be 0");
    MPB_CHECK_ARG(npaths < INT_MAX, "too many paths");
    const int k = subdivisions;
    int64_t nodes_total = 0, bit_words = 0;
    std::vector<ShortcutPath> hp((size_t)npaths + 1);
    for (int64_t q = 0; q < npaths; ++q) {
        const int64_t L = offsets[q + 1] - offsets[q];
        MPB_CHECK_ARG(L >= 1, "offsets must increase: every path needs at least one state");
        MPB_CHECK_ARG(L - 1 <= (MPB200_SHORTCUT_MAX_NODES - 1) / k,
                      "a path has more than MPB200_SHORTCUT_MAX_NODES nodes ((L - 1) subdivisions + 1)");
        const int M = (int)((L - 1) * k + 1);
        hp[q] = ShortcutPath{nodes_total, offsets[q], bit_words, M, (int)L, (M + 31) / 32, 0};
        nodes_total += M;
        bit_words += (int64_t)M * ((M + 31) / 32);
    }
    hp[npaths] = ShortcutPath{nodes_total, offsets[npaths], bit_words, 0, 0, 0, 0};
    if (int rc = shortcut_check_space(o, ss, d)) return rc;

    // scratch: paths | states (the upload) | results | nodes | output rows | best | pred | visibility bits
    const int64_t nstates = offsets[npaths];
    const size_t sz_paths = sizeof(ShortcutPath) * (size_t)(npaths + 1);
    const size_t off_states = align256(sz_paths);
    const size_t off_res = align256(off_states + sizeof(double) * (size_t)nstates * d);
    const size_t off_nodes = align256(off_res + sizeof(ShortcutResult) * (size_t)npaths);
    const size_t off_out = align256(off_nodes + sizeof(double) * (size_t)nodes_total * d);
    const size_t off_best = align256(off_out + sizeof(double) * (size_t)nodes_total * d);
    const size_t off_pred = align256(off_best + sizeof(double) * (size_t)nodes_total);
    const size_t off_bits = align256(off_pred + sizeof(int) * (size_t)nodes_total);
    const size_t total = off_bits + sizeof(uint32_t) * (size_t)bit_words;
    DevBuf scratch;
    if (int rc = scratch.reserve(total)) return rc;
    char *base = scratch.as<char>();
    const ShortcutPath *dpaths = reinterpret_cast<const ShortcutPath *>(base);
    const double *dY = reinterpret_cast<const double *>(base + off_states);
    ShortcutResult *dres = reinterpret_cast<ShortcutResult *>(base + off_res);
    double *dnodes = reinterpret_cast<double *>(base + off_nodes);
    double *dout = reinterpret_cast<double *>(base + off_out);
    double *dbest = reinterpret_cast<double *>(base + off_best);
    int *dpred = reinterpret_cast<int *>(base + off_pred);
    uint32_t *dbits = reinterpret_cast<uint32_t *>(base + off_bits);

    Context &c = ctx();
    cudaStream_t st = c.stream;
    std::vector<char> up(off_res);
    memcpy(up.data(), hp.data(), sz_paths);
    memcpy(up.data() + off_states, states_aos, sizeof(double) * (size_t)nstates * d);
    int rc = 0;
    cudaError_t e = cudaMemcpyAsync(base, up.data(), up.size(), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess)
        rc = shortcut_launch(dpaths, (int)npaths, nodes_total, d, k, dY, o, ss, dnodes, dbits, dbest, dpred, dout, dres);
    std::vector<ShortcutResult> hr((size_t)npaths);
    if (!rc && e == cudaSuccess)
        e = cudaMemcpyAsync(hr.data(), dres, sizeof(ShortcutResult) * (size_t)npaths, cudaMemcpyDeviceToHost, st);
    if (!rc && e == cudaSuccess) e = cudaStreamSynchronize(st);
    for (int64_t q = 0; q < npaths && !rc && e == cudaSuccess; ++q)
        if (hr[q].len <= out_cap)
            e = cudaMemcpyAsync(out_states + q * out_cap * d, dout + hp[q].node0 * d, sizeof(double) * (size_t)hr[q].len * d,
                                cudaMemcpyDeviceToHost, st);
    if (!rc && e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (!rc && e != cudaSuccess) {
        cudaGetLastError();
        rc = fail(MPB200_ECUDA, "shortcutting failed: %s", cudaGetErrorString(e));
    }
    scratch.release();
    if (rc) return rc;
    for (int64_t q = 0; q < npaths; ++q) {
        out_len[q] = hr[q].len;
        costs[q] = hr[q].cost;
        if (pairs) pairs[q] = (int64_t)hp[q].M * (hp[q].M - 1) / 2;
        if (segment_checks) segment_checks[q] = (int64_t)hr[q].checks;
    }
    return MPB200_OK;
}

}  // extern "C"
