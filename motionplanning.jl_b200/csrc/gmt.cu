// gmt.cu -- group-marching FMT* (GMT*) over the device-resident neighbour and validity tables
// (mpb200_gmt_plan; specification in include/mpb200.h and DESIGN.md section 10b).
//
// One persistent cooperative kernel runs the whole planning loop, three grid-wide barriers per iteration:
//   A  split the open list L[p] at thr = min C + w: the group G (status := 2 + it, "in G of iteration it") and the
//      rest (status := 1, appended to L[q]); min of the rest -> minb[q]; smallest goal cost in G -> goalc.
//      The vertices H_new of the previous iteration sit in L[p] with status -1 and become H here.
//   B  one warp per g in G walks column g of DF and claims every unvisited free x with atomicCAS(status, 0, -1):
//      the claim de-duplicates X and keeps x out of H.  When G holds a goal, the smallest goal index of that cost is
//      found instead and the loop ends after the barrier.
//   C  one warp per x in X walks column x of DB over the rows in H (status 1 or 2 + it), shuffle argmin on
//      (cost, position), reads the edge bit of the winner: success writes C[x], A[x] and appends x to L[q]
//      (status stays -1 until the next A, so no x turns into H while other warps still read statuses), failure
//      returns x to W.
// A vertex of an earlier group has status 2 + it' with it' < it, which is neither W nor H: closed, with no pass of its
// own.  Every decision is a min over a set, every counter a sum, so the outputs do not depend on thread order.
#include "common.cuh"
#include "predicates.cuh"
#include <cooperative_groups.h>
#include <climits>
#include <cmath>
#include <cstdlib>
#include <algorithm>

namespace cg = cooperative_groups;

namespace mpb {
namespace {

constexpr int kGmtThreads = 256;
constexpr int kGmtBlocksPerSM = 2;  // 16 warps per SM: enough for the groups of C2 (a few thousand vertices)
constexpr unsigned long long kNone = ~0ULL;

struct GmtCtl {
    unsigned long long minb[2];  // min C bits over the open list of parity p (costs >= 0: integer order = FP order)
    unsigned long long goalc;    // smallest C bits of a goal vertex in G
    unsigned long long checks, checks_inb;
    int nopen[2];                // lengths of the open lists L[0], L[1]
    int ng, nx;                  // |G|, |X|
    int goal;                    // 0-based goal vertex, INT_MAX = none
    int pad;
    // results, written by thread 0 at the end
    long long iterations, expansions, path_len, goal1;
    double cost;
    int solved, pad2;
};

struct GmtArgs {
    const int64_t *fcp, *frv;              // DF
    const int64_t *bcp, *brv;              // DB
    const double *bnz;
    const uint32_t *ebits;                 // DB edge bits
    const uint32_t *pbits;                 // point bits or NULL (all free)
    const uint32_t *gbits;                 // goal mask
    const double *V;                       // d x N
    int N, d, init, inb_on;
    double w;
    double lo[kMaxDim], hi[kMaxDim];
    double *C;
    int64_t *A;
    int *status;                           // 0 W, 1 H, -1 claimed / H_new, 2 + it: in G of iteration it
    int *L0, *L1, *G, *X;
    int64_t *path;
    GmtCtl *ctl;
};

__device__ __forceinline__ bool bit_of(const uint32_t *b, int64_t k) { return (__ldg(b + (k >> 5)) >> (k & 31)) & 1u; }

__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long v) {
    for (int o = 16; o; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// slot of this lane among the lanes of `ballot` (non-zero, whole warp converged) in a list with counter `n`
__device__ __forceinline__ int warp_reserve(int *n, unsigned ballot, int lane) {
    const int leader = __ffs(ballot) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(n, __popc(ballot));
    base = __shfl_sync(0xffffffffu, base, leader);
    return base + __popc(ballot & ((1u << lane) - 1u));
}

__global__ void __launch_bounds__(kGmtThreads) gmt_kernel(const GmtArgs a) {
    cg::grid_group grid = cg::this_grid();
    GmtCtl *ctl = a.ctl;
    const int lane = threadIdx.x & 31;
    const long long gtid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    const long long gwarp = gtid >> 5, nwarps = nthreads >> 5;

    for (long long i = gtid; i < a.N; i += nthreads) {
        a.C[i] = 0.0;
        a.A[i] = 0;
        a.status[i] = i == a.init ? 1 : 0;
    }
    if (gtid == 0) {
        a.L0[0] = a.init;
        ctl->nopen[0] = 1; ctl->nopen[1] = 0;
        ctl->minb[0] = 0; ctl->minb[1] = kNone;  // C[init] = +0.0
        ctl->goalc = kNone; ctl->goal = INT_MAX;
        ctl->ng = 0; ctl->nx = 0;
        ctl->checks = 0; ctl->checks_inb = 0;
    }
    grid.sync();

    long long expansions = 0;
    int it = 0;
    bool solved = false;
    for (;; ++it) {
        const int p = it & 1, q = p ^ 1;
        int *const Lp = p ? a.L1 : a.L0, *const Lq = p ? a.L0 : a.L1;
        const int nopen = ctl->nopen[p];
        if (nopen == 0) break;  // H empty: failed
        const double thr = __dadd_rn(__longlong_as_double((long long)ctl->minb[p]), a.w);
        // ---- A: split L[p] into G and the rest -----------------------------------------------------------
        if (gtid == 0) ctl->nx = 0;
        for (long long i0 = gtid - lane; i0 < nopen; i0 += nthreads) {
            const long long i = i0 + lane;
            int y = -1;
            double c = 0.0;
            if (i < nopen) {
                y = Lp[i];
                c = a.C[y];
            }
            const bool in_g = y >= 0 && c <= thr;
            const bool rest = y >= 0 && !in_g;
            const unsigned bg = __ballot_sync(0xffffffffu, in_g), br = __ballot_sync(0xffffffffu, rest);
            if (bg) {
                const int slot = warp_reserve(&ctl->ng, bg, lane);
                if (in_g) {
                    a.G[slot] = y;
                    a.status[y] = 2 + it;
                }
                const unsigned long long gc = warp_min_u64(in_g && bit_of(a.gbits, y) ? (unsigned long long)__double_as_longlong(c) : kNone);
                if (lane == 0 && gc != kNone) atomicMin(&ctl->goalc, gc);
            }
            if (br) {
                const int slot = warp_reserve(&ctl->nopen[q], br, lane);
                if (rest) {
                    Lq[slot] = y;
                    a.status[y] = 1;
                }
                const unsigned long long m = warp_min_u64(rest ? (unsigned long long)__double_as_longlong(c) : kNone);
                if (lane == 0) atomicMin(&ctl->minb[q], m);
            }
        }
        grid.sync();
        // ---- B: candidates X (or the goal) -------------------------------------------------------------------
        const int ng = ctl->ng;
        const unsigned long long goalc = ctl->goalc;
        if (gtid == 0) {
            ctl->nopen[p] = 0;  // L[p] is consumed; the next iteration's A appends to it
            ctl->minb[p] = kNone;
        }
        for (long long j = gwarp; j < ng; j += nwarps) {
            const int g = a.G[j];
            if (goalc != kNone) {
                if (lane == 0 && bit_of(a.gbits, g) && (unsigned long long)__double_as_longlong(a.C[g]) == goalc)
                    atomicMin(&ctl->goal, g);
                continue;
            }
            const int64_t lo = __ldg(a.fcp + g) - 1, hi = __ldg(a.fcp + g + 1) - 1;
            for (int64_t e0 = lo; e0 < hi; e0 += 32) {
                const int64_t e = e0 + lane;
                bool claim = false;
                int x = 0;
                if (e < hi) {
                    x = (int)(__ldg(a.frv + e) - 1);
                    if (a.status[x] == 0 && (!a.pbits || bit_of(a.pbits, x))) claim = atomicCAS(a.status + x, 0, -1) == 0;
                }
                const unsigned b = __ballot_sync(0xffffffffu, claim);
                if (b) {
                    const int slot = warp_reserve(&ctl->nx, b, lane);
                    if (claim) a.X[slot] = x;
                }
            }
        }
        grid.sync();
        if (goalc != kNone) {
            solved = true;
            break;
        }
        // ---- C: best open parent of every candidate, edge bit, commit ---------------------------------------
        const int nx = ctl->nx;
        if (gtid == 0) {
            expansions += ng;
            ctl->ng = 0;
        }
        const int in_g = 2 + it;
        for (long long j = gwarp; j < nx; j += nwarps) {
            const int x = a.X[j];
            const int64_t lo = __ldg(a.bcp + x) - 1, hi = __ldg(a.bcp + x + 1) - 1;
            double best = INFINITY;
            long long be = LLONG_MAX;
            for (int64_t e = lo + lane; e < hi; e += 32) {
                const int y = (int)(__ldg(a.brv + e) - 1);
                const int s = a.status[y];
                if (s == 1 || s == in_g) {
                    const double c = __dadd_rn(a.C[y], __ldg(a.bnz + e));
                    if (c < best || (c == best && e < be)) {
                        best = c;
                        be = e;
                    }
                }
            }
            for (int o = 16; o; o >>= 1) {
                const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                const long long oe = __shfl_xor_sync(0xffffffffu, be, o);
                if (ob < best || (ob == best && oe < be)) {
                    best = ob;
                    be = oe;
                }
            }
            if (lane != 0) continue;
            if (be == LLONG_MAX) {  // no open neighbour in DB (k-nearest tables): skip x
                a.status[x] = 0;
                continue;
            }
            const int y = (int)(__ldg(a.brv + be) - 1);
            atomicAdd(&ctl->checks, 1ULL);
            if (a.inb_on) {
                bool inb = true;
                for (int k = 0; k < a.d; ++k) {
                    const double v = a.V[(int64_t)y * a.d + k];
                    inb = inb && a.lo[k] <= v && v <= a.hi[k];
                }
                if (inb) atomicAdd(&ctl->checks_inb, 1ULL);
            }
            if (bit_of(a.ebits, be)) {
                a.C[x] = best;
                a.A[x] = y + 1;
                Lq[atomicAdd(&ctl->nopen[q], 1)] = x;
                atomicMin(&ctl->minb[q], (unsigned long long)__double_as_longlong(best));
            } else {
                a.status[x] = 0;
            }
        }
        grid.sync();
    }

    if (gtid == 0) {
        ctl->iterations = it;
        ctl->expansions = expansions;
        ctl->solved = solved;
        if (solved) {
            const int goal = ctl->goal;
            long long n = 1;
            for (int v = goal; v != a.init; v = (int)a.A[v] - 1) ++n;
            long long k = n;
            for (int v = goal;; v = (int)a.A[v] - 1) {
                a.path[--k] = v + 1;
                if (v == a.init) break;
            }
            ctl->path_len = n;
            ctl->goal1 = goal + 1;
            ctl->cost = a.C[goal];
        } else {
            ctl->path_len = 0;
            ctl->goal1 = 0;
            ctl->cost = INFINITY;
        }
    }
}

}  // namespace
}  // namespace mpb

using namespace mpb;

extern "C" {

int mpb200_gmt_plan(const mpb200_samples *s, const mpb200_gmt_desc *desc, mpb200_gmt_result *res, int64_t *path,
                    int64_t path_cap, int64_t *tree, double *costs) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(s != nullptr && desc != nullptr && res != nullptr, "NULL argument");
    MPB_CHECK_ARG(desc->fwd != nullptr && desc->bwd != nullptr, "fwd and bwd tables are required");
    MPB_CHECK_ARG(desc->goal_bits != nullptr, "goal_bits is NULL");
    MPB_CHECK_ARG(path_cap >= 0 && (path != nullptr || path_cap == 0), "path is NULL with path_cap > 0");
    const int64_t N = s->N;
    MPB_CHECK_ARG(N >= 1, "the sample set is empty");
    MPB_CHECK_ARG(desc->init >= 1 && desc->init <= N, "init out of range (1..N)");
    MPB_CHECK_ARG(desc->width >= 0, "width must be a non-negative number");
    MPB_CHECK_ARG(s->d <= kMaxDim, "state dimension out of range");
    for (const mpb200_table *t : {desc->fwd, desc->bwd}) {
        MPB_CHECK_ARG(t->src_serial == s->serial && t->src_N == N && t->src_d == s->d,
                      "a table was not built from this sample set");
        MPB_CHECK_ARG(t->col0 == 0 && t->ncols == N, "a table covers a query range other than [0, N) (sharded tables are not supported)");
    }
    const mpb200_table *B = desc->bwd;
    MPB_CHECK_ARG(B->nnz == 0 || (B->edge_bits_valid && B->edge_bits_nnz == B->nnz),
                  "the backward table has no edge bits for its current contents");
    MPB_CHECK_ARG(!desc->checkpts || s->point_bits_valid, "checkpts needs the point bits of all N samples of this set");
    const mpb200_space_desc *ss = desc->space;
    MPB_CHECK_ARG(!ss || (ss->n == s->d && ss->lo && ss->hi), "space dimension does not match the samples");

    Context &c = ctx();
    cudaStream_t st = c.stream;
    const int64_t gwords = ceil_div(N, 64);
    // scratch: C f64 | A i64 | path i64 | status, L0, L1, G, X i32 | goal bits | control block
    const size_t off_A = sizeof(double) * N, off_path = off_A + sizeof(int64_t) * N;
    const size_t off_i32 = off_path + sizeof(int64_t) * N;
    const size_t off_goal = off_i32 + sizeof(int) * 5 * N + 8 - ((sizeof(int) * 5 * N) & 7);
    const size_t off_ctl = off_goal + sizeof(uint64_t) * gwords;
    DevBuf scratch;
    if (int rc = scratch.reserve(off_ctl + sizeof(GmtCtl))) return rc;
    char *base = scratch.as<char>();
    int *i32 = reinterpret_cast<int *>(base + off_i32);

    GmtArgs a = {};
    a.fcp = desc->fwd->colptr.as<int64_t>(); a.frv = desc->fwd->rowval.as<int64_t>();
    a.bcp = B->colptr.as<int64_t>(); a.brv = B->rowval.as<int64_t>(); a.bnz = B->nzval.as<double>();
    a.ebits = B->edge_bits.as<uint32_t>();
    a.pbits = desc->checkpts ? s->point_bits.as<uint32_t>() : nullptr;
    a.gbits = reinterpret_cast<const uint32_t *>(base + off_goal);
    a.V = s->V.as<double>();
    a.N = (int)N; a.d = s->d; a.init = (int)(desc->init - 1); a.inb_on = ss != nullptr;
    a.w = desc->width;
    for (int k = 0; ss && k < s->d; ++k) a.lo[k] = ss->lo[k], a.hi[k] = ss->hi[k];
    a.C = reinterpret_cast<double *>(base); a.A = reinterpret_cast<int64_t *>(base + off_A);
    a.path = reinterpret_cast<int64_t *>(base + off_path);
    a.status = i32; a.L0 = i32 + N; a.L1 = i32 + 2 * N; a.G = i32 + 3 * N; a.X = i32 + 4 * N;
    a.ctl = reinterpret_cast<GmtCtl *>(base + off_ctl);

    int occ = 0;
    MPB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gmt_kernel, kGmtThreads, 0));
    if (occ < 1) { scratch.release(); return fail(MPB200_ECUDA, "the planning kernel cannot be resident on an SM"); }
    const int max_blocks = occ * c.sm_count;
    static const int env_grid = [] { const char *e = getenv("MPB200_GMT_GRID"); return e ? atoi(e) : 0; }();
    const int blocks = env_grid > 0 ? std::min(env_grid, max_blocks) : std::min(occ, kGmtBlocksPerSM) * c.sm_count;

    int rc = 0;
    cudaError_t e = cudaMemcpyAsync(base + off_goal, desc->goal_bits, sizeof(uint64_t) * gwords, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        phase_bank(MPB200_OP_PLAN);
        phase_mark(0);
        void *args[] = {&a};
        e = cudaLaunchCooperativeKernel((const void *)gmt_kernel, dim3(blocks), dim3(kGmtThreads), args, 0, st);
        c.launches++;
        trace_mark(__FILE__, __LINE__);
        phase_mark(1);
        phases_collect(1);
    }
    GmtCtl h;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h, a.ctl, sizeof(GmtCtl), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && tree) e = cudaMemcpyAsync(tree, a.A, sizeof(int64_t) * N, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && costs) e = cudaMemcpyAsync(costs, a.C, sizeof(double) * N, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess && path && h.path_len > 0 && h.path_len <= path_cap) {
        e = cudaMemcpyAsync(path, a.path, sizeof(int64_t) * h.path_len, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        rc = fail(MPB200_ECUDA, "GMT* planning failed: %s", cudaGetErrorString(e));
    }
    scratch.release();
    if (rc) return rc;
    res->solved = h.solved;
    res->grid_blocks = blocks;
    res->goal = h.goal1;
    res->cost = h.cost;
    res->iterations = h.iterations;
    res->expansions = h.expansions;
    res->checks = (int64_t)h.checks;
    res->checks_in_bounds = (int64_t)h.checks_inb;
    res->path_len = h.path_len;
    return MPB200_OK;
}

}  // extern "C"
