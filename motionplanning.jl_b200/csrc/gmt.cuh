// gmt.cuh -- the GMT* planning kernel (mpb200_gmt_plan / mpb200_gmt_plan_lazy; specification in include/mpb200.h and
// DESIGN.md section 10b), templated on the edge test of step 4.
//
// One persistent cooperative kernel runs the whole planning loop, three grid-wide barriers per iteration:
//   A  split the open list L[p] at thr = min C + w: the group G (status := 2 + it, "in G of iteration it") and the
//      rest (status := 1, appended to L[q]); min of the rest -> minb[q]; smallest goal cost in G -> goalc.
//      The vertices H_new of the previous iteration sit in L[p] with status -1 and become H here.
//   B  one warp per g in G walks column g of DF and claims every unvisited free x with atomicCAS(status, 0, -1):
//      the claim de-duplicates X and keeps x out of H.  When G holds a goal, the smallest goal index of that cost is
//      found instead and the loop ends after the barrier.
//   C  one warp per x in X walks column x of DB over the rows in H (status 1 or 2 + it), shuffle argmin on
//      (cost, position), lane 0 runs the edge test on the winner: success writes C[x], A[x] and appends x to L[q]
//      (status stays -1 until the next A, so no x turns into H while other warps still read statuses), failure
//      returns x to W.
// A vertex of an earlier group has status 2 + it' with it' < it, which is neither W nor H: closed, with no pass of its
// own.  Every decision is a min over a set, every counter a sum, so the outputs do not depend on thread order.
//
// The edge test is a policy: gmt.cu reads the edge bit of the winning entry (table mode); the lazy policies run the
// motion check V[y] -> V[x] of their family (collide.cu, lq.cu, lq_general.cu, cars.cu), each instantiated in the
// translation unit that owns the predicate, and add its segment tests to GmtCtl::segs.
#pragma once
#include "common.cuh"
#include "predicates.cuh"
#include <cooperative_groups.h>
#include <climits>
#include <cmath>

namespace mpb {

constexpr int kGmtThreads = 256;
constexpr int kGmtBlocksPerSM = 2;  // 16 warps per SM: enough for the groups of C2 (a few thousand vertices)
constexpr unsigned long long kGmtNone = ~0ULL;

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
    unsigned long long segs;     // lazy policies: segment tests run by the edge tests
};

struct GmtArgs {
    const int64_t *fcp, *frv;              // DF
    const int64_t *bcp, *brv;              // DB
    const double *bnz;
    const uint32_t *ebits;                 // DB edge bits (table mode)
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

__device__ __forceinline__ bool gmt_bit_of(const uint32_t *b, int64_t k) { return (__ldg(b + (k >> 5)) >> (k & 31)) & 1u; }

__device__ __forceinline__ unsigned long long gmt_warp_min_u64(unsigned long long v) {
    for (int o = 16; o; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// slot of this lane among the lanes of `ballot` (non-zero, whole warp converged) in a list with counter `n`
__device__ __forceinline__ int gmt_warp_reserve(int *n, unsigned ballot, int lane) {
    const int leader = __ffs(ballot) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(n, __popc(ballot));
    base = __shfl_sync(0xffffffffu, base, leader);
    return base + __popc(ballot & ((1u << lane) - 1u));
}

// lazy policies: V[y] and V[x] of the winning entry as N-vectors, and the count of the segment tests run
template <int N>
__device__ __forceinline__ void gmt_endpoints(const GmtArgs &a, int y, int x, double *v, double *w) {
#pragma unroll
    for (int k = 0; k < N; ++k) {
        v[k] = a.V[(int64_t)y * N + k];
        w[k] = a.V[(int64_t)x * N + k];
    }
}
__device__ __forceinline__ void gmt_count_segments(GmtCtl *ctl, int n) {
    if (n) atomicAdd(&ctl->segs, (unsigned long long)n);
}

// Edge: `static constexpr bool kLazy` and `bool operator()(const GmtArgs &, long long e, int y, int x, GmtCtl *)`,
// called by one lane for the winning entry e (row y -> column x) of step 4
template <class Edge>
__global__ void __launch_bounds__(kGmtThreads) gmt_kernel(const GmtArgs a, const Edge edge) {
    namespace cg = cooperative_groups;
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
        ctl->minb[0] = 0; ctl->minb[1] = kGmtNone;  // C[init] = +0.0
        ctl->goalc = kGmtNone; ctl->goal = INT_MAX;
        ctl->ng = 0; ctl->nx = 0;
        ctl->checks = 0; ctl->checks_inb = 0;
        if (Edge::kLazy) ctl->segs = 0;
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
                const int slot = gmt_warp_reserve(&ctl->ng, bg, lane);
                if (in_g) {
                    a.G[slot] = y;
                    a.status[y] = 2 + it;
                }
                const unsigned long long gc =
                    gmt_warp_min_u64(in_g && gmt_bit_of(a.gbits, y) ? (unsigned long long)__double_as_longlong(c) : kGmtNone);
                if (lane == 0 && gc != kGmtNone) atomicMin(&ctl->goalc, gc);
            }
            if (br) {
                const int slot = gmt_warp_reserve(&ctl->nopen[q], br, lane);
                if (rest) {
                    Lq[slot] = y;
                    a.status[y] = 1;
                }
                const unsigned long long m = gmt_warp_min_u64(rest ? (unsigned long long)__double_as_longlong(c) : kGmtNone);
                if (lane == 0) atomicMin(&ctl->minb[q], m);
            }
        }
        grid.sync();
        // ---- B: candidates X (or the goal) -------------------------------------------------------------------
        const int ng = ctl->ng;
        const unsigned long long goalc = ctl->goalc;
        if (gtid == 0) {
            ctl->nopen[p] = 0;  // L[p] is consumed; the next iteration's A appends to it
            ctl->minb[p] = kGmtNone;
        }
        for (long long j = gwarp; j < ng; j += nwarps) {
            const int g = a.G[j];
            if (goalc != kGmtNone) {
                if (lane == 0 && gmt_bit_of(a.gbits, g) && (unsigned long long)__double_as_longlong(a.C[g]) == goalc)
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
                    if (a.status[x] == 0 && (!a.pbits || gmt_bit_of(a.pbits, x))) claim = atomicCAS(a.status + x, 0, -1) == 0;
                }
                const unsigned b = __ballot_sync(0xffffffffu, claim);
                if (b) {
                    const int slot = gmt_warp_reserve(&ctl->nx, b, lane);
                    if (claim) a.X[slot] = x;
                }
            }
        }
        grid.sync();
        if (goalc != kGmtNone) {
            solved = true;
            break;
        }
        // ---- C: best open parent of every candidate, edge test, commit --------------------------------------
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
            if (edge(a, be, y, x, ctl)) {
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

// The cooperative launch of one plan (gmt.cu): grid from the occupancy query (at most kGmtBlocksPerSM blocks per SM,
// MPB200_GMT_GRID=<blocks> overrides, clamped to the co-resident maximum), timed under MPB200_OP_PLAN.
int gmt_launch_kernel(const void *kernel, void **args, int *blocks);

template <class Edge>
int gmt_launch(const GmtArgs &a, const Edge &edge, int *blocks) {
    void *args[] = {const_cast<GmtArgs *>(&a), const_cast<Edge *>(&edge)};
    return gmt_launch_kernel((const void *)gmt_kernel<Edge>, args, blocks);
}

}  // namespace mpb
