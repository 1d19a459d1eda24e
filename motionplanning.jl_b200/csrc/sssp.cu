// sssp.cu -- roadmap-optimal plans (PRM*): exact shortest paths over the device-resident tables and validity bits
// (mpb200_sssp_plan, mpb200_sssp_plan_batch; specification in include/mpb200.h and DESIGN.md section 10d).
//
// One persistent cooperative kernel plans a batch of queries over one roadmap, two phases, no host round trip; a
// single plan is the batch of one.  Query q owns slab q (q * N + v) of D, Dn, tree, h, stamp and pend and its control
// block; the lists hold packed (query, vertex) entries (q << 32 | v, as gmt.cuh), so every phase is one flat loop over
// the union of the queries' work, and all queries share the grid barriers.
//   1  costs.  Near-far relaxation (Davidson et al. 2014; Delta-stepping with one moving threshold per query).  Rounds
//      are synchronous: a round relaxes the out-edges of the vertices of its list L with the costs D as of the round's
//      start and lowers the next costs Dn by atomicMin on the bits (non-negative doubles order like their uint64 bits);
//      the vertices whose cost fell are collected once each in Cl.  After a barrier, each of them takes its new cost and
//      goes to the next L when its cost is <= min(thr, best goal cost) of its query, else it is pending ("far").  When a
//      query's L is empty its threshold moves to min pending cost + Delta (Delta = the largest stored cost of DB, one
//      value for the batch) and its pending vertices below it form L.  The query leaves phase 1 when no pending vertex
//      is at or below its best goal cost.  Every step of the batch is (a) the threshold moves of the queries whose L is
//      empty (skipped grid-uniformly when there is none; the scan covers the slabs of those queries only), then (b) one
//      round of every query still in phase 1.  So each query runs a round in every step until it leaves, its round
//      count is the step at which it leaves, and its sets evolve as in a plan of its own.
//   2  depths and parents.  Level-synchronous BFS over the tight edges inside R = { x : D[x] <= d* } of every query at
//      once: one warp per (q, y) of level L pushes through the out-edges of y and claims each unclaimed tight x with
//      atomicCAS(h, -1, L + 1); then one warp per claimed (q, x) pulls column x of DB and takes the first entry (shuffle
//      argmin on the position) whose row is at depth L and whose edge is tight.  Costs outside R are masked and each
//      query's path is backtracked on the device, one thread per query.
// Out-edges of y are reached through DF: x in column y of DF, then a binary search for row y in column x of DB (rows
// ascending).  That finds every entry of DB with row y because DF holds the transpose of DB (see the header).
// Every FP64 add is __dadd_rn.  The launch goes through gmt_launch_kernel (occupancy sizing, MPB200_GMT_GRID,
// MPB200_OP_PLAN, launch count); the kernel lives here, outside gmt.cuh, so the GMT* kernels are untouched.
#include "gmt.cuh"
#include <vector>

namespace mpb {

namespace {

constexpr unsigned long long kInfBits = 0x7ff0000000000000ULL;  // +inf: above every finite non-negative double

// one per query: written by the host before the launch, then by the kernel
struct SsspCtl {
    unsigned long long goalc;    // smallest D of a goal vertex seen (bits), kInfBits = none
    unsigned long long movemin;  // min pending cost of the last threshold move (bits): thr = movemin + Delta
    unsigned long long scanmin;  // min pending cost of the current threshold move, kGmtNone = none
    unsigned long long nl[2];    // the query's entries of L, by step parity
    unsigned long long nf[2];    // the query's entries of the BFS frontier, by level parity
    long long rounds, levels, reached, path_len, goal1;
    double cost;
    int init, goal, solved;
    int phase1;                  // 1 while the query is in phase 1
};

// batch-wide, written by the host before the launch
struct SsspLists {
    unsigned long long delta;    // largest stored cost of DB (bits)
    unsigned long long nl[2];    // length of L, by step parity
    unsigned long long nc[2];    // length of Cl, by step parity
    unsigned long long nf[2];    // BFS frontier (in L), by level parity
    unsigned long long nx[2];    // BFS claims (in Cl), by level parity
    unsigned long long nfull[2]; // queries with a non-empty L, by step parity
    long long n1;                // queries in phase 1
};

struct SsspArgs {
    const int64_t *fcp, *frv;              // DF
    const int64_t *bcp, *brv;              // DB
    const double *bnz;
    const uint32_t *ebits;                 // DB edge bits
    const uint32_t *pbits;                 // point bits or NULL (all free)
    const uint32_t *gbits;                 // goal masks, nq x gstride words
    int N, nq;
    int64_t gstride;                       // 32-bit words per goal mask
    int64_t nnz;
    int64_t path_cap;                      // row length of path (0: no paths)
    unsigned long long *D, *Dn;            // nq x N each; Dn ends as the output costs
    int64_t *tree;                         // nq x N, 1-based parents
    int *h;                                // nq x N, BFS depth, -1 = none
    int *stamp;                            // nq x N, last round + 1 in which the vertex joined Cl
    int *pend;                             // nq x N, 1 = cost fell above the threshold, not yet relaxed
    unsigned long long *L, *Cl;            // packed entries, nq x N each: round / frontier list, changed / claimed list
    int64_t *path;                         // nq x path_cap, 1-based
    SsspCtl *ctl;                          // nq
    SsspLists *lists;
};

__device__ __forceinline__ bool sssp_bit(const uint32_t *b, int64_t k) { return (__ldg(b + (k >> 5)) >> (k & 31)) & 1u; }

// first entry of column x of DB whose row is y (0-based), or the end of the column when there is none
__device__ __forceinline__ int64_t sssp_find(const SsspArgs &a, int x, int y, int64_t *end) {
    int64_t lo = __ldg(a.bcp + x) - 1, hi = __ldg(a.bcp + x + 1) - 1;
    *end = hi;
    const int64_t key = (int64_t)y + 1;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(a.brv + mid) < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// f(x, e) for every graph edge y -> x (entry e of DB) reached from lane `lane` of the warp walking column y of DF
template <class F>
__device__ __forceinline__ void sssp_out_edges(const SsspArgs &a, int y, int lane, F f) {
    const int64_t lo = __ldg(a.fcp + y) - 1, hi = __ldg(a.fcp + y + 1) - 1;
    for (int64_t k = lo + lane; k < hi; k += 32) {
        const int x = (int)(__ldg(a.frv + k) - 1);
        if (x == y || (a.pbits && !sssp_bit(a.pbits, x))) continue;
        int64_t end;
        for (int64_t e = sssp_find(a, x, y, &end); e < end && __ldg(a.brv + e) == (int64_t)y + 1; ++e)
            if (sssp_bit(a.ebits, e)) f(x, e);
    }
}

__device__ __forceinline__ double sssp_cost(unsigned long long b) { return __longlong_as_double((long long)b); }
__device__ __forceinline__ unsigned long long sssp_bits(double c) { return (unsigned long long)__double_as_longlong(c); }

__global__ void __launch_bounds__(kGmtThreads, kGmtBlocksPerSM) sssp_kernel(const SsspArgs a) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    SsspCtl *const ctl = a.ctl;
    SsspLists *const lists = a.lists;
    const int lane = threadIdx.x & 31;
    const long long gtid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    const long long gwarp = gtid >> 5, nwarps = nthreads >> 5;
    // per-query bookkeeping runs on the last threads of the grid, which the list loops (from thread 0 up) leave idle
    const long long rtid = nthreads - 1 - gtid;
    const int N = a.N, nq = a.nq;

    // ---- set-up: state of every vertex of every query, Delta --------------------------------------------------
    for (int q = 0; q < nq; ++q) {
        const int init = ctl[q].init;
        const int64_t base = (int64_t)q * N;
        for (long long i = gtid; i < N; i += nthreads) {
            const unsigned long long c = i == init ? 0ULL : kInfBits;
            a.D[base + i] = c;
            a.Dn[base + i] = c;
            a.h[base + i] = i == init ? 0 : -1;
            a.tree[base + i] = 0;
            a.stamp[base + i] = 0;
            a.pend[base + i] = 0;
        }
    }
    {
        unsigned long long m = 0;
        for (long long e = gtid; e < a.nnz; e += nthreads) m = max(m, sssp_bits(__ldg(a.bnz + e)));
        for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0 && m) atomicMax(&lists->delta, m);
    }
    for (long long q = gtid; q < nq; q += nthreads) a.L[q] = gmt_entry((int)q, ctl[q].init);  // L = [init] per query
    grid.sync();

    // ---- phase 1: costs ---------------------------------------------------------------------------------------
    const double delta = sssp_cost(lists->delta);
    int step = 0;
    for (;; ++step) {
        const int p = step & 1;
        if (lists->n1 > (long long)lists->nfull[p]) {
            // (a) threshold moves of the queries in phase 1 whose L is empty: min pending cost at or below the best
            // goal cost, over their slabs only
            for (int q = 0; q < nq; ++q) {
                if (!ctl[q].phase1 || ctl[q].nl[p]) continue;
                const unsigned long long goalc = ctl[q].goalc;
                const int64_t base = (int64_t)q * N;
                unsigned long long m = kGmtNone;
                for (long long i = gtid; i < N; i += nthreads)
                    if (a.pend[base + i]) {
                        const unsigned long long c = a.D[base + i];
                        if (c <= goalc) m = min(m, c);
                    }
                m = gmt_warp_min_u64(m);
                if (lane == 0 && m != kGmtNone) atomicMin(&ctl[q].scanmin, m);
            }
            grid.sync();
            // a query with nothing pending at or below d* leaves phase 1: every cost of its R is final
            for (long long q = rtid; q < nq; q += nthreads) {
                if (!ctl[q].phase1 || ctl[q].nl[p]) continue;
                const unsigned long long m = ctl[q].scanmin;
                if (m == kGmtNone) {
                    ctl[q].phase1 = 0;
                    ctl[q].rounds = step;
                    atomicAdd((unsigned long long *)&lists->n1, ~0ULL);
                } else {
                    ctl[q].movemin = m;
                }
            }
            for (int q = 0; q < nq; ++q) {  // (its phase1 flag may have been cleared already: then m is none)
                if (!ctl[q].phase1 || ctl[q].nl[p]) continue;
                const unsigned long long m = ctl[q].scanmin;
                if (m == kGmtNone) continue;
                const unsigned long long bound = min(sssp_bits(__dadd_rn(sssp_cost(m), delta)), ctl[q].goalc);
                const int64_t base = (int64_t)q * N;
                for (long long i0 = gtid - lane; i0 < N; i0 += nthreads) {
                    const long long i = i0 + lane;
                    const bool take = i < N && a.pend[base + i] && a.D[base + i] <= bound;
                    const unsigned b = __ballot_sync(0xffffffffu, take);
                    if (b) {
                        const long long slot = gmt_warp_reserve(&lists->nl[p], b, lane);
                        if (take) {
                            a.pend[base + i] = 0;
                            a.L[slot] = gmt_entry(q, (int)i);
                        }
                    }
                }
            }
            grid.sync();
        }
        if (lists->n1 == 0) break;
        // (b) one round of every query in phase 1: relax the out-edges of L with the costs of the round's start
        const long long nl = (long long)lists->nl[p];
        if (gtid == 0) {
            lists->nl[p ^ 1] = 0;
            lists->nfull[p ^ 1] = 0;
        }
        for (long long q = rtid; q < nq; q += nthreads) {
            ctl[q].nl[p ^ 1] = 0;
            ctl[q].scanmin = kGmtNone;
        }
        const int tag = step + 1;  // the query's own round + 1: every query in phase 1 has run a round in every step
        for (long long j = gwarp; j < nl; j += nwarps) {
            const unsigned long long ent = a.L[j];
            const int q = (int)(ent >> 32), y = (int)(unsigned)ent;
            const int64_t base = (int64_t)q * N;
            const uint32_t *const gb = a.gbits + q * a.gstride;
            const double c = sssp_cost(a.D[base + y]);
            sssp_out_edges(a, y, lane, [&](int x, int64_t e) {
                const unsigned long long nd = sssp_bits(__dadd_rn(c, __ldg(a.bnz + e)));
                if (nd < *(volatile unsigned long long *)(a.Dn + base + x) && nd < atomicMin(a.Dn + base + x, nd)) {
                    if (sssp_bit(gb, x)) atomicMin(&ctl[q].goalc, nd);
                    if (atomicExch(a.stamp + base + x, tag) != tag)
                        a.Cl[atomicAdd(&lists->nc[p], 1ULL)] = gmt_entry(q, x);
                }
            });
        }
        grid.sync();
        // the vertices whose cost fell take it; near ones form the next L, far ones are pending
        const long long nc = (long long)lists->nc[p];
        if (gtid == 0) lists->nc[p ^ 1] = 0;
        for (long long i0 = gtid - lane; i0 < nc; i0 += nthreads) {
            const long long i = i0 + lane;
            unsigned long long ent = 0;
            int q = 0;
            bool near = false;
            if (i < nc) {
                ent = a.Cl[i];
                q = (int)(ent >> 32);
                const int64_t v = (int64_t)q * N + (int)(unsigned)ent;
                const unsigned long long thr = sssp_bits(__dadd_rn(sssp_cost(ctl[q].movemin), delta));
                const unsigned long long c = a.Dn[v];
                a.D[v] = c;
                near = c <= min(thr, ctl[q].goalc);
                a.pend[v] = !near;
            }
            const unsigned b = __ballot_sync(0xffffffffu, near);
            if (b) {
                const long long slot = gmt_warp_reserve(&lists->nl[p ^ 1], b, lane);
                if (near) a.L[slot] = ent;
                // per-query lengths: one pass per query present in the warp
                for (unsigned left = b; left;) {
                    const int leader = __ffs(left) - 1;
                    const int gq = __shfl_sync(0xffffffffu, q, leader);
                    const unsigned m = __ballot_sync(0xffffffffu, near && q == gq);
                    left &= ~m;
                    if (lane == leader && atomicAdd(&ctl[gq].nl[p ^ 1], (unsigned long long)__popc(m)) == 0)
                        atomicAdd(&lists->nfull[p ^ 1], 1ULL);
                }
            }
        }
        grid.sync();
    }

    // ---- phase 2: depths and parents over the tight edges inside R of every query ------------------------------
    int level = 0;
    for (;; ++level) {
        const int par = level & 1;
        const long long nf = (long long)lists->nf[par];
        for (long long q = rtid; q < nq; q += nthreads) {  // per query: frontier size into |R|; first empty level
            const unsigned long long n = ctl[q].nf[par];
            if (n) ctl[q].reached += (long long)n;
            else if (ctl[q].levels < 0) ctl[q].levels = level;
            ctl[q].nf[par ^ 1] = 0;
        }
        if (nf == 0) break;
        if (gtid == 0) lists->nf[par ^ 1] = 0;
        for (long long j = gwarp; j < nf; j += nwarps) {  // push: claim the unclaimed tight out-neighbours in R
            // depth 0 is the init of query j (L still holds phase 1's last entries)
            const unsigned long long ent = level ? a.L[j] : gmt_entry((int)j, ctl[j].init);
            const int q = (int)(ent >> 32), y = (int)(unsigned)ent;
            const int64_t base = (int64_t)q * N;
            const unsigned long long dstar = ctl[q].goalc;
            const unsigned long long rmax = dstar == kInfBits ? kInfBits - 1 : dstar;  // failed: R = every reachable
            const double c = sssp_cost(a.D[base + y]);
            sssp_out_edges(a, y, lane, [&](int x, int64_t e) {
                const unsigned long long dx = a.D[base + x];
                if (dx <= rmax && a.h[base + x] == -1 && sssp_bits(__dadd_rn(c, __ldg(a.bnz + e))) == dx &&
                    atomicCAS(a.h + base + x, -1, level + 1) == -1)
                    a.Cl[atomicAdd(&lists->nx[par], 1ULL)] = gmt_entry(q, x);
            });
        }
        grid.sync();
        const long long nx = (long long)lists->nx[par];
        if (gtid == 0) lists->nx[par ^ 1] = 0;
        for (long long j = gwarp; j < nx; j += nwarps) {  // pull: the first tight entry of column x from depth `level`
            const unsigned long long ent = a.Cl[j];
            const int q = (int)(ent >> 32), x = (int)(unsigned)ent;
            const int64_t base = (int64_t)q * N;
            const unsigned long long dx = a.D[base + x];
            const int64_t lo = __ldg(a.bcp + x) - 1, hi = __ldg(a.bcp + x + 1) - 1;
            long long be = LLONG_MAX;
            for (int64_t e = lo + lane; e < hi && be == LLONG_MAX; e += 32) {
                const int y = (int)(__ldg(a.brv + e) - 1);
                if (y != x && a.h[base + y] == level && sssp_bit(a.ebits, e) &&
                    sssp_bits(__dadd_rn(sssp_cost(a.D[base + y]), __ldg(a.bnz + e))) == dx)
                    be = e;
            }
            for (int o = 16; o; o >>= 1) be = min(be, __shfl_xor_sync(0xffffffffu, be, o));
            if (lane != 0) continue;
            if (be == LLONG_MAX) {  // cannot happen (the claim came through a tight entry); released for safety
                a.h[base + x] = -1;
                continue;
            }
            a.tree[base + x] = __ldg(a.brv + be);
            a.L[atomicAdd(&lists->nf[par ^ 1], 1ULL)] = ent;
            atomicAdd(&ctl[q].nf[par ^ 1], 1ULL);
        }
        grid.sync();
    }

    // ---- outputs: costs masked to R, the goal, the path ---------------------------------------------------------
    for (int q = 0; q < nq; ++q) {
        const int64_t base = (int64_t)q * N;
        const uint32_t *const gb = a.gbits + q * a.gstride;
        const unsigned long long dstar = ctl[q].goalc;
        const unsigned long long rmax = dstar == kInfBits ? kInfBits - 1 : dstar;
        for (long long i = gtid; i < N; i += nthreads) {
            const unsigned long long c = a.D[base + i];
            const bool in_r = c <= rmax;
            a.Dn[base + i] = in_r ? c : kInfBits;
            if (in_r && c == dstar && sssp_bit(gb, i)) atomicMin(&ctl[q].goal, (int)i);
        }
    }
    grid.sync();
    for (long long q = gtid; q < nq; q += nthreads) {  // one thread per query
        SsspCtl *const cq = ctl + q;
        const int init = cq->init;
        const int64_t base = q * (int64_t)N;
        const unsigned long long dstar = cq->goalc;
        const int goal = sssp_bit(a.gbits + q * a.gstride, init) ? init : cq->goal;
        if (dstar != kInfBits) {
            const long long n = (long long)a.h[base + goal] + 1;
            if (n <= a.path_cap) {
                int64_t *const path = a.path + q * a.path_cap;
                long long k = n;
                for (int v = goal;; v = (int)a.tree[base + v] - 1) {
                    path[--k] = v + 1;
                    if (v == init) break;
                }
            }
            cq->solved = 1;
            cq->path_len = n;
            cq->goal1 = goal + 1;
            cq->cost = sssp_cost(dstar);
        } else {
            cq->path_len = 0;
            cq->goal1 = 0;
            cq->cost = INFINITY;
        }
    }
}

}  // namespace

// A single plan is the batch of one query.
static int sssp_plan(const mpb200_samples *s, const mpb200_gmt_desc *descs, int64_t nq, mpb200_sssp_result *res,
                     int64_t *paths, int64_t path_cap, int64_t *trees, double *costs) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(s != nullptr && descs != nullptr && res != nullptr, "NULL argument");
    MPB_CHECK_ARG(nq >= 1, "a batch needs at least one query");
    const mpb200_gmt_desc *desc = descs;  // the fields every query shares
    MPB_CHECK_ARG(desc->fwd != nullptr && desc->bwd != nullptr, "fwd and bwd tables are required");
    for (int64_t q = 0; q < nq; ++q) {
        const mpb200_gmt_desc &dq = descs[q];
        MPB_CHECK_ARG(dq.fwd == desc->fwd && dq.bwd == desc->bwd && !dq.checkpts == !desc->checkpts,
                      "the queries of a batch must share fwd, bwd and checkpts");
        MPB_CHECK_ARG(dq.goal_bits != nullptr, "goal_bits is NULL");
    }
    MPB_CHECK_ARG(path_cap >= 0 && (paths != nullptr || path_cap == 0), "path is NULL with path_cap > 0");
    const int64_t N = s->N;
    MPB_CHECK_ARG(N >= 1, "the sample set is empty");
    for (int64_t q = 0; q < nq; ++q) MPB_CHECK_ARG(descs[q].init >= 1 && descs[q].init <= N, "init out of range (1..N)");
    if (int rc = gmt_check_roadmap(s, desc, true)) return rc;
    const mpb200_table *B = desc->bwd;

    Context &c = ctx();
    cudaStream_t st = c.stream;
    const int64_t gwords = ceil_div(N, 64);
    const int64_t pcap = std::min(path_cap, N);  // no path is longer than N
    // scratch: D, Dn u64 | tree i64 | L, Cl u64 | paths i64 | lists | control blocks | goal masks | h, stamp, pend i32,
    // the N-sized arrays nq times; the 8-byte fields come first, so they stay aligned whatever N
    // (MPB200_SSSP_BATCH_BYTES_PER_QUERY in include/mpb200.h, plus the 96 bytes of lists)
    static_assert(sizeof(SsspCtl) == 120, "MPB200_SSSP_BATCH_BYTES_PER_QUERY counts 120 bytes of control block");
    static_assert(sizeof(SsspLists) == 96, "MPB200_SSSP_BYTES counts 96 bytes of lists");
    const size_t per_query = (size_t)N * (5 * 8 + 3 * 4) + sizeof(int64_t) * pcap + sizeof(SsspCtl) +
                             sizeof(uint64_t) * gwords;
    if (nq > INT_MAX || (size_t)nq > (SIZE_MAX - sizeof(SsspLists)) / per_query)
        return fail(MPB200_ENOMEM, "a batch of %lld queries over %lld samples does not fit in device memory",
                    (long long)nq, (long long)N);
    const size_t nN = (size_t)nq * N;
    const size_t off_Dn = sizeof(uint64_t) * nN, off_tree = 2 * off_Dn, off_L = off_tree + sizeof(int64_t) * nN;
    const size_t off_path = off_L + 2 * sizeof(uint64_t) * nN;
    const size_t off_lists = off_path + sizeof(int64_t) * nq * pcap;
    const size_t off_ctl = off_lists + sizeof(SsspLists), off_goal = off_ctl + sizeof(SsspCtl) * nq;
    const size_t off_i32 = off_goal + sizeof(uint64_t) * gwords * nq;
    DevBuf scratch;
    if (int rc = scratch.reserve(off_i32 + sizeof(int) * 3 * nN)) return rc;
    char *base = scratch.as<char>();

    // lists, control blocks and goal masks start as the host writes them: one copy
    std::vector<char> init(off_i32 - off_lists);
    SsspLists *hl = reinterpret_cast<SsspLists *>(init.data());
    hl->nl[0] = (unsigned long long)nq;     // L = [init] per query
    hl->nf[0] = (unsigned long long)nq;     // the BFS frontiers of depth 0: the inits
    hl->nfull[0] = (unsigned long long)nq;
    hl->n1 = nq;
    SsspCtl *hc = reinterpret_cast<SsspCtl *>(init.data() + (off_ctl - off_lists));
    for (int64_t q = 0; q < nq; ++q) {
        hc[q].goalc = kInfBits;
        hc[q].scanmin = kGmtNone;
        hc[q].nl[0] = 1;
        hc[q].nf[0] = 1;
        hc[q].levels = -1;
        hc[q].init = (int)(descs[q].init - 1);
        hc[q].goal = INT_MAX;
        hc[q].phase1 = 1;
        const uint64_t *g64 = descs[q].goal_bits;
        memcpy(init.data() + (off_goal - off_lists) + sizeof(uint64_t) * gwords * q, g64, sizeof(uint64_t) * gwords);
        if ((g64[(descs[q].init - 1) >> 6] >> ((descs[q].init - 1) & 63)) & 1) hc[q].goalc = 0;  // init is a goal
    }

    SsspArgs a = {};
    a.fcp = desc->fwd->colptr.as<int64_t>(); a.frv = desc->fwd->rowval.as<int64_t>();
    a.bcp = B->colptr.as<int64_t>(); a.brv = B->rowval.as<int64_t>(); a.bnz = B->nzval.as<double>();
    a.ebits = B->edge_bits.as<uint32_t>();
    a.pbits = desc->checkpts ? s->point_bits.as<uint32_t>() : nullptr;
    a.gbits = reinterpret_cast<const uint32_t *>(base + off_goal);
    a.gstride = 2 * gwords;
    a.N = (int)N; a.nq = (int)nq; a.nnz = B->nnz; a.path_cap = pcap;
    a.D = reinterpret_cast<unsigned long long *>(base);
    a.Dn = reinterpret_cast<unsigned long long *>(base + off_Dn);
    a.tree = reinterpret_cast<int64_t *>(base + off_tree);
    a.L = reinterpret_cast<unsigned long long *>(base + off_L);
    a.Cl = a.L + nN;
    a.path = pcap ? reinterpret_cast<int64_t *>(base + off_path) : nullptr;
    int *i32 = reinterpret_cast<int *>(base + off_i32);
    a.h = i32; a.stamp = i32 + nN; a.pend = i32 + 2 * nN;
    a.lists = reinterpret_cast<SsspLists *>(base + off_lists);
    a.ctl = reinterpret_cast<SsspCtl *>(base + off_ctl);

    int blocks = 0, rc = 0;
    cudaError_t e = cudaMemcpyAsync(base + off_lists, init.data(), init.size(), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        void *args[] = {&a};
        rc = gmt_launch_kernel((const void *)sssp_kernel, args, &blocks);
    }
    if (rc) {
        scratch.release();
        return rc;
    }
    std::vector<SsspCtl> h(nq);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h.data(), a.ctl, sizeof(SsspCtl) * nq, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && trees) e = cudaMemcpyAsync(trees, a.tree, sizeof(int64_t) * nN, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && costs) e = cudaMemcpyAsync(costs, a.Dn, sizeof(double) * nN, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    bool copied = false;
    for (int64_t q = 0; q < nq && e == cudaSuccess; ++q) {  // the rows that fit, path_len entries each
        if (h[q].path_len > 0 && h[q].path_len <= pcap) {
            e = cudaMemcpyAsync(paths + q * path_cap, a.path + q * pcap, sizeof(int64_t) * h[q].path_len,
                                cudaMemcpyDeviceToHost, st);
            copied = true;
        }
    }
    if (e == cudaSuccess && copied) e = cudaStreamSynchronize(st);
    scratch.release();
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(MPB200_ECUDA, "PRM* planning failed: %s", cudaGetErrorString(e));
    }
    for (int64_t q = 0; q < nq; ++q) {
        res[q].solved = h[q].solved;
        res[q].grid_blocks = blocks;
        res[q].goal = h[q].goal1;
        res[q].cost = h[q].cost;
        res[q].path_len = h[q].path_len;
        res[q].rounds = h[q].rounds;
        res[q].levels = h[q].levels;
        res[q].reached = h[q].reached;
    }
    return MPB200_OK;
}

}  // namespace mpb

using namespace mpb;

extern "C" {

int mpb200_sssp_plan(const mpb200_samples *s, const mpb200_gmt_desc *desc, mpb200_sssp_result *res, int64_t *path,
                     int64_t path_cap, int64_t *tree, double *costs) {
    return sssp_plan(s, desc, 1, res, path, path_cap, tree, costs);
}

int mpb200_sssp_plan_batch(const mpb200_samples *s, const mpb200_gmt_desc *descs, int64_t nq,
                           mpb200_sssp_result *res, int64_t *paths, int64_t path_cap, int64_t *trees, double *costs) {
    return sssp_plan(s, descs, nq, res, paths, path_cap, trees, costs);
}

}  // extern "C"
