// gmt.cuh -- the GMT* planning kernel (mpb200_gmt_plan / _lazy / _batch; specification in include/mpb200.h and
// DESIGN.md section 10b), templated on the edge test of step 4.
//
// One persistent cooperative kernel runs the whole planning loop of a batch of queries over one roadmap, three
// grid-wide barriers per iteration shared by every query.  Each list holds (query, vertex) entries of all queries, so
// every phase is one flat loop over the union of their work; a single plan is the batch of one.
//   A  split the open list L[p] at thr = min C + w of the entry's query: the group G (status := 2 + it, "in G of
//      iteration it") and the rest (status := 1, appended to L[q]); min of the rest -> minb[q]; smallest goal cost in
//      G -> goalc.  A query whose open set is empty fails here.
//      The vertices H_new of the previous iteration sit in L[p] with status -1 and become H here.
//   B  one warp per g in G walks column g of DF and claims every unvisited free x with atomicCAS(status, 0, -1):
//      the claim de-duplicates X and keeps x out of H.  When G holds a goal, the smallest goal index of that cost is
//      found instead and the query ends; the loop ends after the barrier when no query is left.
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

// one per query: written by the host before the launch (init, w, the initial values below), then by the kernel
struct GmtCtl {
    unsigned long long minb[2];  // min C bits over the query's entries of L[p] (costs >= 0: integer order = FP order);
                                 // kGmtNone = none, so the query's open set of parity p is empty
    unsigned long long goalc;    // smallest C bits of a goal vertex in G
    unsigned long long checks, checks_inb;
    unsigned long long segs;     // lazy policies: segment tests run by the edge tests
    double w;                    // width
    int init;                    // 0-based
    int goal;                    // 0-based goal vertex, INT_MAX = none
    int done;                    // 1 once the query has solved or failed: its list entries are dropped
    // results
    long long iterations, expansions, path_len, goal1;
    double cost;
    int solved, pad;
};

// batch-wide list lengths, written by the host before the launch
struct GmtLists {
    unsigned long long nopen[2];  // L[0], L[1]
    unsigned long long ng, nx;    // G, X
    int nactive;                  // queries not yet done
    int pad;
};

// A list entry packs (query, vertex): q << 32 | v.  Query q's state lives in slab q of C, A and status (q * N + v).
struct GmtArgs {
    const int64_t *fcp, *frv;              // DF
    const int64_t *bcp, *brv;              // DB
    const double *bnz;
    const uint32_t *ebits;                 // DB edge bits (table mode)
    const uint32_t *pbits;                 // point bits or NULL (all free)
    const uint32_t *gbits;                 // goal masks, nq x gstride words
    const double *V;                       // d x N
    int N, d, nq, inb_on;
    int64_t gstride;                       // 32-bit words per goal mask
    int64_t path_cap;                      // row length of path (0: no paths)
    double lo[kMaxDim], hi[kMaxDim];
    double *C;                             // nq x N
    int64_t *A;                            // nq x N
    int *status;                           // nq x N: 0 W, 1 H, -1 claimed / H_new, 2 + it: in G of iteration it
    unsigned long long *L0, *L1, *G, *X;   // packed entries, nq x N each
    int64_t *path;                         // nq x path_cap, 1-based
    GmtCtl *ctl;                           // nq
    GmtLists *lists;
};

__device__ __forceinline__ bool gmt_bit_of(const uint32_t *b, int64_t k) { return (__ldg(b + (k >> 5)) >> (k & 31)) & 1u; }

__device__ __forceinline__ unsigned long long gmt_warp_min_u64(unsigned long long v) {
    for (int o = 16; o; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// slot of this lane among the lanes of `ballot` (non-zero, whole warp converged) in a list with counter `n`
__device__ __forceinline__ long long gmt_warp_reserve(unsigned long long *n, unsigned ballot, int lane) {
    const int leader = __ffs(ballot) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(n, (unsigned long long)__popc(ballot));
    base = __shfl_sync(0xffffffffu, base, leader);
    return (long long)(base + __popc(ballot & ((1u << lane) - 1u)));
}

__device__ __forceinline__ unsigned long long gmt_entry(int q, int v) {
    return (unsigned long long)(unsigned)q << 32 | (unsigned)v;
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
// called by one lane for the winning entry e (row y -> column x) of step 4, with the control block of its query.
// Queries march in lockstep: iteration `it` is global, each query's phases touch only its own slab and control block,
// and a query that has ended contributes no list entries, so its outputs are those of a plan of its own.
template <class Edge>
__global__ void __launch_bounds__(kGmtThreads) gmt_kernel(const GmtArgs a, const Edge edge) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    GmtCtl *const ctl = a.ctl;
    GmtLists *const lists = a.lists;
    const int lane = threadIdx.x & 31;
    const long long gtid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    const long long gwarp = gtid >> 5, nwarps = nthreads >> 5;
    // the per-query bookkeeping of each phase runs on the last threads of the grid, which the list loops (handed out
    // from thread 0 up) leave idle unless the lists are long: its dependent loads stay off the phase's critical path
    const long long rtid = nthreads - 1 - gtid;
    const int64_t N = a.N;

    for (int q = 0; q < a.nq; ++q) {
        const int init = ctl[q].init;
        double *const C = a.C + q * N;
        int64_t *const A = a.A + q * N;
        int *const status = a.status + q * N;
        for (long long i = gtid; i < N; i += nthreads) {
            C[i] = 0.0;
            A[i] = 0;
            status[i] = i == init ? 1 : 0;
        }
    }
    for (long long q = gtid; q < a.nq; q += nthreads) a.L0[q] = gmt_entry((int)q, ctl[q].init);
    grid.sync();

    int it = 0;
    for (;; ++it) {
        const int p = it & 1, pq = p ^ 1;
        unsigned long long *const Lp = p ? a.L1 : a.L0, *const Lq = p ? a.L0 : a.L1;
        const long long nopen = (long long)lists->nopen[p];
        if (nopen == 0) break;  // every open set empty: the queries still active fail
        // ---- A: split L[p] into G and the rest, per query at thr = min C + w ----------------------------------
        if (gtid == 0) lists->nx = 0;
        for (long long q = rtid; q < a.nq; q += nthreads) {
            if (!ctl[q].done && ctl[q].minb[p] == kGmtNone) {  // H empty: failed
                ctl[q].done = 1;
                ctl[q].iterations = it;
                atomicSub(&lists->nactive, 1);
            }
        }
        for (long long i0 = gtid - lane; i0 < nopen; i0 += nthreads) {
            const long long i = i0 + lane;
            unsigned long long ent = 0;
            int q = 0, y = 0;
            bool live = false;
            double c = 0.0, thr = 0.0;
            if (i < nopen) {  // the four loads depend on the entry only, so they are in flight together
                ent = Lp[i];
                q = (int)(ent >> 32);
                y = (int)(unsigned)ent;
                live = !ctl[q].done;
                c = a.C[q * N + y];
                thr = __dadd_rn(__longlong_as_double((long long)ctl[q].minb[p]), ctl[q].w);
            }
            const bool in_g = live && c <= thr;
            const bool rest = live && !in_g;
            const unsigned bg = __ballot_sync(0xffffffffu, in_g), br = __ballot_sync(0xffffffffu, rest);
            if (bg) {
                const long long slot = gmt_warp_reserve(&lists->ng, bg, lane);
                if (in_g) {
                    a.G[slot] = ent;
                    a.status[q * N + y] = 2 + it;
                }
            }
            if (br) {
                const long long slot = gmt_warp_reserve(&lists->nopen[pq], br, lane);
                if (rest) {
                    Lq[slot] = ent;
                    a.status[q * N + y] = 1;
                }
            }
            // per-query sums and minima: one pass per query present in the warp
            for (unsigned pend = bg | br; pend;) {
                const int leader = __ffs(pend) - 1;
                const int gq = __shfl_sync(0xffffffffu, q, leader);
                const bool mine = (in_g || rest) && q == gq;
                const unsigned m = __ballot_sync(0xffffffffu, mine);
                pend &= ~m;
                if (m & bg) {
                    const unsigned long long gc = gmt_warp_min_u64(
                        mine && in_g && gmt_bit_of(a.gbits + gq * a.gstride, y) ? (unsigned long long)__double_as_longlong(c)
                                                                               : kGmtNone);
                    if (lane == leader && gc != kGmtNone) atomicMin(&ctl[gq].goalc, gc);
                }
                if (m & br) {
                    const unsigned long long rm =
                        gmt_warp_min_u64(mine && rest ? (unsigned long long)__double_as_longlong(c) : kGmtNone);
                    if (lane == leader) atomicMin(&ctl[gq].minb[pq], rm);
                }
            }
        }
        grid.sync();
        // ---- B: candidates X (or the goal) -------------------------------------------------------------------
        const long long ng = (long long)lists->ng;
        if (gtid == 0) lists->nopen[p] = 0;  // L[p] is consumed; the next iteration's A appends to it
        for (long long q = rtid; q < a.nq; q += nthreads) {
            ctl[q].minb[p] = kGmtNone;
            if (!ctl[q].done && ctl[q].goalc != kGmtNone) {  // G holds a goal: solved
                ctl[q].done = 1;
                ctl[q].solved = 1;
                ctl[q].iterations = it;
                atomicSub(&lists->nactive, 1);
            }
        }
        for (long long j = gwarp; j < ng; j += nwarps) {
            const unsigned long long ent = a.G[j];
            const int q = (int)(ent >> 32), g = (int)(unsigned)ent;
            const int64_t base = q * N;
            const unsigned long long goalc = ctl[q].goalc;
            const int64_t lo = __ldg(a.fcp + g) - 1, hi = __ldg(a.fcp + g + 1) - 1;  // in flight with goalc
            if (goalc != kGmtNone) {
                if (lane == 0 && gmt_bit_of(a.gbits + q * a.gstride, g) &&
                    (unsigned long long)__double_as_longlong(a.C[base + g]) == goalc)
                    atomicMin(&ctl[q].goal, g);
                continue;
            }
            for (int64_t e0 = lo; e0 < hi; e0 += 32) {
                const int64_t e = e0 + lane;
                bool claim = false;
                int x = 0;
                if (e < hi) {
                    x = (int)(__ldg(a.frv + e) - 1);
                    if (a.status[base + x] == 0 && (!a.pbits || gmt_bit_of(a.pbits, x)))
                        claim = atomicCAS(a.status + base + x, 0, -1) == 0;
                }
                const unsigned b = __ballot_sync(0xffffffffu, claim);
                if (b) {
                    const long long slot = gmt_warp_reserve(&lists->nx, b, lane);
                    if (claim) a.X[slot] = gmt_entry(q, x);
                }
            }
        }
        grid.sync();
        if (lists->nactive == 0) break;
        // ---- C: best open parent of every candidate, edge test, commit --------------------------------------
        const long long nx = (long long)lists->nx;
        if (gtid == 0) lists->ng = 0;
        const int in_g = 2 + it;
        for (long long j = gwarp; j < nx; j += nwarps) {
            const unsigned long long ent = a.X[j];
            const int q = (int)(ent >> 32), x = (int)(unsigned)ent;
            const int64_t base = q * N;
            const int64_t lo = __ldg(a.bcp + x) - 1, hi = __ldg(a.bcp + x + 1) - 1;
            double best = INFINITY;
            long long be = LLONG_MAX;
            for (int64_t e = lo + lane; e < hi; e += 32) {
                const int y = (int)(__ldg(a.brv + e) - 1);
                const int s = a.status[base + y];
                if (s == 1 || s == in_g) {
                    const double c = __dadd_rn(a.C[base + y], __ldg(a.bnz + e));
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
                a.status[base + x] = 0;
                continue;
            }
            const int y = (int)(__ldg(a.brv + be) - 1);
            atomicAdd(&ctl[q].checks, 1ULL);
            if (a.inb_on) {
                bool inb = true;
                for (int k = 0; k < a.d; ++k) {
                    const double v = a.V[(int64_t)y * a.d + k];
                    inb = inb && a.lo[k] <= v && v <= a.hi[k];
                }
                if (inb) atomicAdd(&ctl[q].checks_inb, 1ULL);
            }
            // only q, x, y and best live across the edge test: the lazy policies need every register they can get
            if (edge(a, be, y, x, ctl + q)) {
                a.C[q * N + x] = best;
                a.A[q * N + x] = y + 1;
                Lq[atomicAdd(&lists->nopen[pq], 1ULL)] = gmt_entry(q, x);
                atomicMin(&ctl[q].minb[pq], (unsigned long long)__double_as_longlong(best));
            } else {
                a.status[q * N + x] = 0;
            }
        }
        grid.sync();
    }

    // expansions: a vertex that was in G of iteration it' keeps status 2 + it', so the groups a query expanded are the
    // vertices of its slab with 2 <= status < 2 + its iterations (a solving group has status 2 + iterations)
    for (int q = 0; q < a.nq; ++q) {
        const int end = 2 + (ctl[q].done ? (int)ctl[q].iterations : it);
        const int *const status = a.status + q * N;
        int n = 0;
        for (long long i = gtid; i < N; i += nthreads) {
            const int s = status[i];
            n += s >= 2 && s < end;
        }
        n = __reduce_add_sync(0xffffffffu, n);
        if (lane == 0 && n) atomicAdd((unsigned long long *)&ctl[q].expansions, (unsigned long long)n);
    }
    // results and paths: one thread per query
    for (long long q = gtid; q < a.nq; q += nthreads) {
        GmtCtl *const cq = ctl + q;
        if (!cq->done) cq->iterations = it;  // its open set was empty when the loop ended
        if (cq->solved) {
            const int goal = cq->goal, init = cq->init;
            const int64_t *const A = a.A + q * N;
            long long n = 1;
            for (int v = goal; v != init; v = (int)A[v] - 1) ++n;
            if (n <= a.path_cap) {
                int64_t *const path = a.path + q * a.path_cap;
                long long k = n;
                for (int v = goal;; v = (int)A[v] - 1) {
                    path[--k] = v + 1;
                    if (v == init) break;
                }
            }
            cq->path_len = n;
            cq->goal1 = goal + 1;
            cq->cost = a.C[q * N + goal];
        } else {
            cq->path_len = 0;
            cq->goal1 = 0;
            cq->cost = INFINITY;
        }
    }
}

// The cooperative launch of one batch (gmt.cu): grid from the occupancy query (at most kGmtBlocksPerSM blocks per SM,
// MPB200_GMT_GRID=<blocks> overrides, clamped to the co-resident maximum), timed under MPB200_OP_PLAN.
int gmt_launch_kernel(const void *kernel, void **args, int *blocks);

template <class Edge>
int gmt_launch(const GmtArgs &a, const Edge &edge, int *blocks) {
    void *args[] = {const_cast<GmtArgs *>(&a), const_cast<Edge *>(&edge)};
    return gmt_launch_kernel((const void *)gmt_kernel<Edge>, args, blocks);
}

}  // namespace mpb
