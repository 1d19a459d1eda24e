// sssp.cu -- roadmap-optimal plans (PRM*): exact shortest paths over the device-resident tables and validity bits
// (mpb200_sssp_plan; specification in include/mpb200.h and DESIGN.md section 10d).
//
// One persistent cooperative kernel, two phases, no host round trip:
//   1  costs.  Near-far relaxation (Davidson et al. 2014; Delta-stepping with one moving threshold).  Rounds are
//      synchronous: a round relaxes the out-edges of the vertices of its list L with the costs D as of the round's start
//      and lowers the next costs Dn by atomicMin on the bits (non-negative doubles order like their uint64 bits); the
//      vertices whose cost fell are collected once each in Cl.  After a barrier, each of them takes its new cost and
//      goes to the next L when its cost is <= min(thr, best goal cost), else it is pending ("far").  When L is empty the
//      threshold moves to min pending cost + Delta (Delta = the largest stored cost of DB) and the pending vertices
//      below it form L.  The search ends when no pending vertex is at or below the best goal cost.  Since every round
//      is a function of the previous round's sets, so are the round count and every cost.
//   2  depths and parents.  Level-synchronous BFS over the tight edges inside R = { x : D[x] <= d* }: one warp per
//      vertex y of level L pushes through the out-edges of y and claims each unclaimed tight x with atomicCAS(h, -1,
//      L + 1); then one warp per claimed x pulls column x of DB and takes the first entry (shuffle argmin on the
//      position) whose row is at depth L and whose edge is tight.  Costs outside R are masked and the path is
//      backtracked on the device.
// Out-edges of y are reached through DF: x in column y of DF, then a binary search for row y in column x of DB (rows
// ascending).  That finds every entry of DB with row y because DF holds the transpose of DB (see the header).
// Every FP64 add is __dadd_rn.  The launch goes through gmt_launch_kernel (occupancy sizing, MPB200_GMT_GRID,
// MPB200_OP_PLAN, launch count); the kernel lives here, outside gmt.cuh, so the GMT* kernels are untouched.
#include "gmt.cuh"
#include <vector>

namespace mpb {

namespace {

constexpr unsigned long long kInfBits = 0x7ff0000000000000ULL;  // +inf: above every finite non-negative double

struct SsspCtl {
    unsigned long long delta;       // largest stored cost of DB (bits)
    unsigned long long goalc;       // smallest D of a goal vertex seen (bits), kInfBits = none
    unsigned long long scanmin[2];  // min pending cost of a threshold move, by move parity
    unsigned long long nl[2];       // length of L, by round parity
    unsigned long long nc[2];       // length of Cl, by round parity
    unsigned long long nf[2];       // BFS frontier (in L), by level parity
    unsigned long long nx[2];       // BFS claims (in Cl), by level parity
    long long rounds, levels, reached, path_len, goal1;
    double cost;
    int init, goal, solved, pad;
};

struct SsspArgs {
    const int64_t *fcp, *frv;              // DF
    const int64_t *bcp, *brv;              // DB
    const double *bnz;
    const uint32_t *ebits;                 // DB edge bits
    const uint32_t *pbits;                 // point bits or NULL (all free)
    const uint32_t *gbits;                 // goal mask
    int N;
    int64_t nnz;
    int64_t path_cap;
    unsigned long long *D, *Dn;            // N each; Dn ends as the output costs
    int64_t *tree;                         // N, 1-based parents
    int *h;                                // N, BFS depth, -1 = none
    int *stamp;                            // N, last round + 1 in which the vertex joined Cl
    int *pend;                             // N, 1 = cost fell above the threshold, not yet relaxed
    int *L, *Cl;                           // N each: round / frontier list, changed / claimed list
    int64_t *path;
    SsspCtl *ctl;
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
    const int lane = threadIdx.x & 31;
    const long long gtid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    const long long gwarp = gtid >> 5, nwarps = nthreads >> 5;
    const int N = a.N, init = ctl->init;

    // ---- set-up: state of every vertex, Delta ---------------------------------------------------------------
    for (long long i = gtid; i < N; i += nthreads) {
        const unsigned long long c = i == init ? 0ULL : kInfBits;
        a.D[i] = c;
        a.Dn[i] = c;
        a.h[i] = i == init ? 0 : -1;
        a.tree[i] = 0;
        a.stamp[i] = 0;
        a.pend[i] = 0;
    }
    {
        unsigned long long m = 0;
        for (long long e = gtid; e < a.nnz; e += nthreads) m = max(m, sssp_bits(__ldg(a.bnz + e)));
        for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0 && m) atomicMax(&ctl->delta, m);
    }
    if (gtid == 0) a.L[0] = init;
    grid.sync();

    // ---- phase 1: costs ---------------------------------------------------------------------------------------
    const double delta = sssp_cost(ctl->delta);
    unsigned long long thr = sssp_bits(__dadd_rn(0.0, delta));
    int round = 0, moves = 0;
    for (;; ++round) {
        const int p = round & 1;
        long long nl = (long long)ctl->nl[p];
        if (nl == 0) {  // move the threshold: min pending cost at or below the best goal cost, + Delta
            const unsigned long long goalc = ctl->goalc;
            unsigned long long m = kGmtNone;
            for (long long i = gtid; i < N; i += nthreads)
                if (a.pend[i]) {
                    const unsigned long long c = a.D[i];
                    if (c <= goalc) m = min(m, c);
                }
            m = gmt_warp_min_u64(m);
            if (lane == 0 && m != kGmtNone) atomicMin(&ctl->scanmin[moves & 1], m);
            grid.sync();
            m = ctl->scanmin[moves & 1];
            if (m == kGmtNone) break;  // nothing pending at or below d*: every cost in R is final
            thr = sssp_bits(__dadd_rn(sssp_cost(m), delta));
            const unsigned long long bound = min(thr, goalc);
            if (gtid == 0) ctl->scanmin[(moves + 1) & 1] = kGmtNone;
            for (long long i0 = gtid - lane; i0 < N; i0 += nthreads) {
                const long long i = i0 + lane;
                const bool take = i < N && a.pend[i] && a.D[i] <= bound;
                const unsigned b = __ballot_sync(0xffffffffu, take);
                if (b) {
                    const long long slot = gmt_warp_reserve(&ctl->nl[p], b, lane);
                    if (take) {
                        a.pend[i] = 0;
                        a.L[slot] = (int)i;
                    }
                }
            }
            ++moves;
            grid.sync();
            nl = (long long)ctl->nl[p];
        }
        // relax the out-edges of L with the costs of the round's start
        if (gtid == 0) ctl->nl[p ^ 1] = 0;
        const int tag = round + 1;
        for (long long j = gwarp; j < nl; j += nwarps) {
            const int y = a.L[j];
            const double c = sssp_cost(a.D[y]);
            sssp_out_edges(a, y, lane, [&](int x, int64_t e) {
                const unsigned long long nd = sssp_bits(__dadd_rn(c, __ldg(a.bnz + e)));
                if (nd < *(volatile unsigned long long *)(a.Dn + x) && nd < atomicMin(a.Dn + x, nd)) {
                    if (sssp_bit(a.gbits, x)) atomicMin(&ctl->goalc, nd);
                    if (atomicExch(a.stamp + x, tag) != tag) a.Cl[atomicAdd(&ctl->nc[p], 1ULL)] = x;
                }
            });
        }
        grid.sync();
        // the vertices whose cost fell take it; near ones form the next L, far ones are pending
        const long long nc = (long long)ctl->nc[p];
        if (gtid == 0) ctl->nc[p ^ 1] = 0;
        const unsigned long long bound = min(thr, ctl->goalc);
        for (long long i0 = gtid - lane; i0 < nc; i0 += nthreads) {
            const long long i = i0 + lane;
            int x = 0;
            bool near = false;
            if (i < nc) {
                x = a.Cl[i];
                const unsigned long long c = a.Dn[x];
                a.D[x] = c;
                near = c <= bound;
                a.pend[x] = !near;
            }
            const unsigned b = __ballot_sync(0xffffffffu, near);
            if (b) {
                const long long slot = gmt_warp_reserve(&ctl->nl[p ^ 1], b, lane);
                if (near) a.L[slot] = x;
            }
        }
        grid.sync();
    }

    // ---- phase 2: depths and parents over the tight edges inside R --------------------------------------------
    const unsigned long long dstar = ctl->goalc;
    const unsigned long long rmax = dstar == kInfBits ? kInfBits - 1 : dstar;  // failed: R = every reachable vertex
    int level = 0;
    long long reached = 0;
    for (;; ++level) {
        const int q = level & 1;
        const long long nf = (long long)ctl->nf[q];
        if (nf == 0) break;
        reached += nf;
        if (gtid == 0) ctl->nf[q ^ 1] = 0;
        for (long long j = gwarp; j < nf; j += nwarps) {  // push: claim the unclaimed tight out-neighbours in R
            const int y = level ? a.L[j] : init;  // L still holds phase 1's last list at depth 0
            const double c = sssp_cost(a.D[y]);
            sssp_out_edges(a, y, lane, [&](int x, int64_t e) {
                const unsigned long long dx = a.D[x];
                if (dx <= rmax && a.h[x] == -1 && sssp_bits(__dadd_rn(c, __ldg(a.bnz + e))) == dx &&
                    atomicCAS(a.h + x, -1, level + 1) == -1)
                    a.Cl[atomicAdd(&ctl->nx[q], 1ULL)] = x;
            });
        }
        grid.sync();
        const long long nx = (long long)ctl->nx[q];
        if (gtid == 0) ctl->nx[q ^ 1] = 0;
        for (long long j = gwarp; j < nx; j += nwarps) {  // pull: the first tight entry of column x from depth `level`
            const int x = a.Cl[j];
            const unsigned long long dx = a.D[x];
            const int64_t lo = __ldg(a.bcp + x) - 1, hi = __ldg(a.bcp + x + 1) - 1;
            long long be = LLONG_MAX;
            for (int64_t e = lo + lane; e < hi && be == LLONG_MAX; e += 32) {
                const int y = (int)(__ldg(a.brv + e) - 1);
                if (y != x && a.h[y] == level && sssp_bit(a.ebits, e) &&
                    sssp_bits(__dadd_rn(sssp_cost(a.D[y]), __ldg(a.bnz + e))) == dx)
                    be = e;
            }
            for (int o = 16; o; o >>= 1) be = min(be, __shfl_xor_sync(0xffffffffu, be, o));
            if (lane != 0) continue;
            if (be == LLONG_MAX) {  // cannot happen (the claim came through a tight entry); released for safety
                a.h[x] = -1;
                continue;
            }
            a.tree[x] = __ldg(a.brv + be);
            a.L[atomicAdd(&ctl->nf[q ^ 1], 1ULL)] = x;
        }
        grid.sync();
    }

    // ---- outputs: costs masked to R, the goal, the path --------------------------------------------------------
    for (long long i = gtid; i < N; i += nthreads) {
        const unsigned long long c = a.D[i];
        const bool in_r = c <= rmax;
        a.Dn[i] = in_r ? c : kInfBits;
        if (in_r && c == dstar && sssp_bit(a.gbits, i)) atomicMin(&ctl->goal, (int)i);
    }
    grid.sync();
    if (gtid == 0) {
        ctl->rounds = round;
        ctl->levels = level;
        ctl->reached = reached;
        const int goal = sssp_bit(a.gbits, init) ? init : ctl->goal;
        if (dstar != kInfBits) {
            const long long n = (long long)a.h[goal] + 1;
            if (n <= a.path_cap) {
                long long k = n;
                for (int v = goal;; v = (int)a.tree[v] - 1) {
                    a.path[--k] = v + 1;
                    if (v == init) break;
                }
            }
            ctl->solved = 1;
            ctl->path_len = n;
            ctl->goal1 = goal + 1;
            ctl->cost = sssp_cost(dstar);
        } else {
            ctl->path_len = 0;
            ctl->goal1 = 0;
            ctl->cost = INFINITY;
        }
    }
}

}  // namespace

static int sssp_plan(const mpb200_samples *s, const mpb200_gmt_desc *desc, mpb200_sssp_result *res, int64_t *path,
                     int64_t path_cap, int64_t *tree, double *costs) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(s != nullptr && desc != nullptr && res != nullptr, "NULL argument");
    MPB_CHECK_ARG(desc->fwd != nullptr && desc->bwd != nullptr, "fwd and bwd tables are required");
    MPB_CHECK_ARG(desc->goal_bits != nullptr, "goal_bits is NULL");
    MPB_CHECK_ARG(path_cap >= 0 && (path != nullptr || path_cap == 0), "path is NULL with path_cap > 0");
    const int64_t N = s->N;
    MPB_CHECK_ARG(N >= 1, "the sample set is empty");
    MPB_CHECK_ARG(desc->init >= 1 && desc->init <= N, "init out of range (1..N)");
    if (int rc = gmt_check_roadmap(s, desc, true)) return rc;
    const mpb200_table *B = desc->bwd;

    Context &c = ctx();
    cudaStream_t st = c.stream;
    const int64_t gwords = ceil_div(N, 64);
    const int64_t pcap = std::min(path_cap, N);
    // scratch: D, Dn u64 | tree, path i64 | control block | goal mask | h, stamp, pend, L, Cl i32; the 8-byte fields
    // come first, so they stay aligned whatever N (MPB200_SSSP_BYTES in include/mpb200.h)
    static_assert(sizeof(SsspCtl) == 160, "MPB200_SSSP_BYTES counts 160 bytes of control block");
    const size_t off_Dn = sizeof(uint64_t) * N, off_tree = 2 * off_Dn, off_path = off_tree + sizeof(int64_t) * N;
    const size_t off_ctl = off_path + sizeof(int64_t) * pcap;
    const size_t off_goal = off_ctl + sizeof(SsspCtl);
    const size_t off_i32 = off_goal + sizeof(uint64_t) * gwords;
    DevBuf scratch;
    if (int rc = scratch.reserve(off_i32 + sizeof(int) * 5 * N)) return rc;
    char *base = scratch.as<char>();

    std::vector<char> init(sizeof(SsspCtl) + sizeof(uint64_t) * gwords);
    SsspCtl *hc = reinterpret_cast<SsspCtl *>(init.data());
    hc->goalc = kInfBits;
    hc->scanmin[0] = hc->scanmin[1] = kGmtNone;
    hc->nl[0] = 1;  // L = [init]
    hc->nf[0] = 1;  // the BFS frontier of depth 0: init
    hc->init = (int)(desc->init - 1);
    hc->goal = INT_MAX;
    memcpy(init.data() + sizeof(SsspCtl), desc->goal_bits, sizeof(uint64_t) * gwords);
    const uint64_t *g64 = desc->goal_bits;
    if ((g64[(desc->init - 1) >> 6] >> ((desc->init - 1) & 63)) & 1) hc->goalc = 0;  // init is a goal: d* = 0

    SsspArgs a = {};
    a.fcp = desc->fwd->colptr.as<int64_t>(); a.frv = desc->fwd->rowval.as<int64_t>();
    a.bcp = B->colptr.as<int64_t>(); a.brv = B->rowval.as<int64_t>(); a.bnz = B->nzval.as<double>();
    a.ebits = B->edge_bits.as<uint32_t>();
    a.pbits = desc->checkpts ? s->point_bits.as<uint32_t>() : nullptr;
    a.gbits = reinterpret_cast<const uint32_t *>(base + off_goal);
    a.N = (int)N; a.nnz = B->nnz; a.path_cap = pcap;
    a.D = reinterpret_cast<unsigned long long *>(base);
    a.Dn = reinterpret_cast<unsigned long long *>(base + off_Dn);
    a.tree = reinterpret_cast<int64_t *>(base + off_tree);
    a.path = pcap ? reinterpret_cast<int64_t *>(base + off_path) : nullptr;
    int *i32 = reinterpret_cast<int *>(base + off_i32);
    a.h = i32; a.stamp = i32 + N; a.pend = i32 + 2 * N; a.L = i32 + 3 * N; a.Cl = i32 + 4 * N;
    a.ctl = reinterpret_cast<SsspCtl *>(base + off_ctl);

    int blocks = 0, rc = 0;
    cudaError_t e = cudaMemcpyAsync(base + off_ctl, init.data(), init.size(), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        void *args[] = {&a};
        rc = gmt_launch_kernel((const void *)sssp_kernel, args, &blocks);
    }
    if (rc) {
        scratch.release();
        return rc;
    }
    SsspCtl h;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h, a.ctl, sizeof(SsspCtl), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && tree) e = cudaMemcpyAsync(tree, a.tree, sizeof(int64_t) * N, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && costs) e = cudaMemcpyAsync(costs, a.Dn, sizeof(double) * N, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess && h.path_len > 0 && h.path_len <= pcap) {
        e = cudaMemcpyAsync(path, a.path, sizeof(int64_t) * h.path_len, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    scratch.release();
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(MPB200_ECUDA, "PRM* planning failed: %s", cudaGetErrorString(e));
    }
    res->solved = h.solved;
    res->grid_blocks = blocks;
    res->goal = h.goal1;
    res->cost = h.cost;
    res->path_len = h.path_len;
    res->rounds = h.rounds;
    res->levels = h.levels;
    res->reached = h.reached;
    return MPB200_OK;
}

}  // namespace mpb

using namespace mpb;

extern "C" int mpb200_sssp_plan(const mpb200_samples *s, const mpb200_gmt_desc *desc, mpb200_sssp_result *res,
                                int64_t *path, int64_t path_cap, int64_t *tree, double *costs) {
    return sssp_plan(s, desc, res, path, path_cap, tree, costs);
}
