// lq.cu -- K5 (ControlNN: all-pairs linear-quadratic steering-cost neighbour tables) and
// K9 (swept-trajectory edge checks along the optimal LQ trajectory) for double-integrator systems.
//
// Replaces helper_data_structures(V, ::LinearQuadratic) (linearquadratic.jl:68-77): the column-
// batched dense steer_pairwise (:196-225: dcost(r) > 0 prefilter, per-candidate safeguarded
// Newton topt_newton :175-190, keep cost <= r) followed by the inball filter
// (nearneighbors.jl:165-177), producing both DSF (column v = costs FROM v) and DSB (column v =
// costs INTO v); and is_free_motion(v, w, CC, SS) with collision_waypoints of :85-88
// (5 states along x(s), statespaces.jl:153-158).
//
// The reference's SymPy closures reduce, for A=[0 I;0 0], B=[0;I], c=0, to
//   cost(t) = t + alpha/t^3 - beta/t^2 + gamma/t
// (see oracle/lq.c; pinned by tests/golden/lq_di2.json).  Operation order here is identical to
// the oracle's, every operation an explicit _rn intrinsic (no FMA), so tables are bit-identical.
//
// Layout: one thread per query column (its state in registers, both directions evaluated against
// the same staged sample), samples streamed through shared memory in tiles and read by
// broadcast; rows come out in ascending index order, so no sort is needed.
#include "common.cuh"
#include "predicates.cuh"
#include "scan.cuh"
#include "gmt.cuh"

namespace mpb {

struct LqDev {
    int scalar_R;
    double R[9];
};
struct Abg { double alpha, beta, gamma; };

// alpha, beta, gamma in the oracle's order (oracle/lq.c: lq_abg)
template <int D>
__device__ __forceinline__ Abg lq_abg(const LqDev &L, const double *x0, const double *x1) {
    double dp[D], sv[D];
    const double *v0 = x0 + D, *v1 = x1 + D;
#pragma unroll
    for (int i = 0; i < D; ++i) { dp[i] = dsub(x1[i], x0[i]); sv[i] = dadd(v0[i], v1[i]); }
    double a = 0.0, b = 0.0, g = 0.0;
#pragma unroll
    for (int i = 0; i < D; ++i) {
        double Rdp, Rv0, Rv1;
        if (L.scalar_R) {  // R = rho I: the off-diagonal products are exact zeros
            Rdp = dmul(L.R[0], dp[i]); Rv0 = dmul(L.R[0], v0[i]); Rv1 = dmul(L.R[0], v1[i]);
        } else {
            Rdp = 0.0; Rv0 = 0.0; Rv1 = 0.0;
#pragma unroll
            for (int j = 0; j < D; ++j) {
                Rdp = dadd(Rdp, dmul(L.R[i * D + j], dp[j]));
                Rv0 = dadd(Rv0, dmul(L.R[i * D + j], v0[j]));
                Rv1 = dadd(Rv1, dmul(L.R[i * D + j], v1[j]));
            }
        }
        a = dadd(a, dmul(dp[i], Rdp));
        b = dadd(b, dmul(sv[i], Rdp));
        g = dadd(g, dadd(dadd(dmul(v0[i], Rv0), dmul(v0[i], Rv1)), dmul(v1[i], Rv1)));
    }
    Abg k = {dmul(12.0, a), dmul(12.0, b), dmul(4.0, g)};
    return k;
}
// Both directions of one pair at once for the stage-1 prefilter: kF = lq_abg(x, y), kB = lq_abg(y, x), bit for
// bit.  Swapping the roles negates dp = x1 - x0 exactly, so every product with it is negated exactly as well:
// alpha (quadratic in dp) is unchanged and beta changes sign; sv = v0 + v1 is commutative.  Only gamma has a
// different operation order in the two directions and is evaluated twice.
template <int D>
__device__ __forceinline__ void lq_abg_both(const LqDev &L, const double *x, const double *y, Abg *kF, Abg *kB) {
    double dp[D], sv[D];
    const double *vx = x + D, *vy = y + D;
#pragma unroll
    for (int i = 0; i < D; ++i) { dp[i] = dsub(y[i], x[i]); sv[i] = dadd(vx[i], vy[i]); }
    double a = 0.0, b = 0.0, gF = 0.0, gB = 0.0;
#pragma unroll
    for (int i = 0; i < D; ++i) {
        double Rdp, Rvx, Rvy;
        if (L.scalar_R) {
            Rdp = dmul(L.R[0], dp[i]); Rvx = dmul(L.R[0], vx[i]); Rvy = dmul(L.R[0], vy[i]);
        } else {
            Rdp = 0.0; Rvx = 0.0; Rvy = 0.0;
#pragma unroll
            for (int j = 0; j < D; ++j) {
                Rdp = dadd(Rdp, dmul(L.R[i * D + j], dp[j]));
                Rvx = dadd(Rvx, dmul(L.R[i * D + j], vx[j]));
                Rvy = dadd(Rvy, dmul(L.R[i * D + j], vy[j]));
            }
        }
        a = dadd(a, dmul(dp[i], Rdp));
        b = dadd(b, dmul(sv[i], Rdp));
        gF = dadd(gF, dadd(dadd(dmul(vx[i], Rvx), dmul(vx[i], Rvy)), dmul(vy[i], Rvy)));  // v0 = vx, v1 = vy
        gB = dadd(gB, dadd(dadd(dmul(vy[i], Rvy), dmul(vy[i], Rvx)), dmul(vx[i], Rvx)));  // v0 = vy, v1 = vx
    }
    const double alpha = dmul(12.0, a), beta = dmul(12.0, b);
    kF->alpha = alpha; kF->beta = beta;  kF->gamma = dmul(4.0, gF);
    kB->alpha = alpha; kB->beta = -beta; kB->gamma = dmul(4.0, gB);
}
__device__ __forceinline__ double lq_cost(const Abg &k, double t) {
    const double it = ddiv(1.0, t), it2 = dmul(it, it), it3 = dmul(it2, it);
    return dadd(t, dadd(dsub(dmul(k.alpha, it3), dmul(k.beta, it2)), dmul(k.gamma, it)));
}
__device__ __forceinline__ double lq_dcost(const Abg &k, double t) {
    const double it = ddiv(1.0, t), it2 = dmul(it, it), it3 = dmul(it2, it);
    return dadd(1.0, dsub(dsub(dmul(dmul(2.0, k.beta), it3), dmul(dmul(3.0, k.alpha), dmul(it3, it))),
                          dmul(k.gamma, it2)));
}
__device__ __forceinline__ double lq_ddcost(const Abg &k, double t) {
    const double it = ddiv(1.0, t), it2 = dmul(it, it), it3 = dmul(it2, it);
    return dadd(dsub(dmul(dmul(12.0, k.alpha), dmul(it3, it2)), dmul(dmul(6.0, k.beta), dmul(it2, it2))),
                dmul(dmul(2.0, k.gamma), it3));
}
// linearquadratic.jl:175-190 (same 200-iteration safety cap as the oracle; never reached)
__device__ __forceinline__ double lq_topt_newton(const Abg &k, double tm) {
    const double tol = 1e-6;
    double b = tm;
    if (lq_dcost(k, b) < 0) return tm;
    double a = ddiv(tm, 100.0);
    while (lq_dcost(k, a) > 0) a = ddiv(a, 2.0);
    double t = ddiv(tm, 2.0);
    double cdval = lq_dcost(k, t);
    int it = 0;
    while (fabs(cdval) > tol && fabs(dsub(a, b)) > tol) {
        t = dsub(t, ddiv(cdval, lq_ddcost(k, t)));
        if (t < a || t > b) t = ddiv(dadd(a, b), 2.0);
        cdval = lq_dcost(k, t);
        if (cdval > 0) b = t; else a = t;
        if (++it >= 200) break;
    }
    return t;
}
template <int D>
__device__ __forceinline__ bool same_state(const double *x0, const double *x1) {
    bool same = true;
#pragma unroll
    for (int i = 0; i < 2 * D; ++i) same = same && (x0[i] == x1[i]);
    return same;
}
// steer(L, x0, x1, r): linearquadratic.jl:191-195
template <int D>
__device__ __forceinline__ void lq_steer(const LqDev &L, const double *x0, const double *x1, double r, double *cost,
                                         double *topt) {
    if (same_state<D>(x0, x1)) { *cost = 0.0; *topt = 0.0; return; }
    const Abg k = lq_abg<D>(L, x0, x1);
    const double t = lq_topt_newton(k, r);
    *cost = lq_cost(k, t);
    *topt = t;
}
// x(x0, x1, t, s): cubic Hermite in Horner form (oracle/lq.c: orc_lq_state)
template <int D>
__device__ __forceinline__ void lq_state(const double *x0, const double *x1, double t, double s, double *out) {
    const double it = ddiv(1.0, t), it2 = dmul(it, it), it3 = dmul(it2, it);
    const double *v0 = x0 + D, *v1 = x1 + D;
#pragma unroll
    for (int i = 0; i < D; ++i) {
        const double dp = dsub(x1[i], x0[i]);
        const double c2 = dsub(dmul(dmul(3.0, dp), it2), dmul(dadd(dmul(2.0, v0[i]), v1[i]), it));
        const double c3 = dsub(dmul(dadd(v0[i], v1[i]), it2), dmul(dmul(2.0, dp), it3));
        out[i] = dadd(dmul(dadd(dmul(dadd(dmul(c3, s), c2), s), v0[i]), s), x0[i]);
        out[D + i] = dadd(dmul(dadd(dmul(dmul(3.0, c3), s), dmul(2.0, c2)), s), v0[i]);
    }
}

// one ordered pair x0 -> x1: is it a stored neighbour, and at what cost
template <int D>
__device__ __forceinline__ bool lq_pair(const LqDev &L, const double *x0, const double *x1, double r, double *cost) {
    const Abg k = lq_abg<D>(L, x0, x1);
    if (!(lq_dcost(k, r) > 0)) return false;  // cands = cd .> 0, linearquadratic.jl:213
    double c;
    if (same_state<D>(x0, x1)) c = 0.0;       // :192 (duplicate states)
    else c = lq_cost(k, lq_topt_newton(k, r));
    *cost = c;
    return c <= r;                            // :221
}

// FP32 stage-1 constants of one table build (lq_prefilter)
struct LqPre {
    double center[3];  // positions are centred before the FP32 conversion (dp is translation invariant)
    float R[9];        // D x D row-major
    float c2, c3, c4;  // 4/r^2, 24/r^3, 36/r^4
    float neg_delta;   // keep a pair when the FP32 dcost(r) exceeds this (< 0)
    float r2, delta2;  // ... and a (16 g - r^2) - 12 b^2 <= delta2 (second necessary condition, see lq_prefilter)
};

constexpr int kLqThreads = 128;
constexpr int kLqTile = 128;

// K5.  MODE 0: per-column counts for both directions; MODE 1: rows + costs into the CSC arrays;
// MODE 2: ONE sweep that counts and appends every neighbour (index, cost) to the column's slab
// (capacity `cap` per direction), finished by lq_slab_to_csc -- the all-pairs work runs once.
//
// Two stages per warp.  Stage 1 is uniform: every lane evaluates alpha/beta/gamma and the reference's
// candidate test dcost(r) > 0 (linearquadratic.jl:213) for its own query against the staged sample, both
// directions; a fraction of a percent of the pairs survive.  Running the safeguarded Newton right there
// left 7 of 32 lanes busy (ncu, profiles/r1/lq_inball_ncu_summary.txt: 61% of stall samples on fixed-latency
// dependencies of the few active lanes).  Survivors are therefore pushed, in lane order, into a per-warp ring
// (owner lane | direction | sample index), and stage 2 runs whenever 32 are waiting: lane e takes item e,
// reads the owner's state from shared memory and the sample from global memory, redoes alpha/beta/gamma in the
// same operation order (bit-identical), runs topt_newton + cost, and the accepted ones are emitted to their
// owner's column.  Items of one (owner, direction) enter the ring in ascending sample order and leave it in
// FIFO order; inside a batch the slot is the owner's running count plus the number of accepted earlier
// peers (match.any + ballot), so rows still come out ascending without a sort.
template <int D, int MODE>
__global__ void __launch_bounds__(kLqThreads, 4)  // 100 registers, no spills (the default heuristic spilled the stage-1 state)
lq_inball_kernel(const double *__restrict__ V, int64_t N, int64_t q0, int64_t nq, LqDev L, LqPre P, double r,
                 int *__restrict__ countsF, int *__restrict__ countsB, const int64_t *__restrict__ colptrF,
                 const int64_t *__restrict__ colptrB, int64_t *__restrict__ rowvalF, double *__restrict__ nzvalF,
                 int64_t *__restrict__ rowvalB, double *__restrict__ nzvalB, int cap, int *__restrict__ slabF_j,
                 double *__restrict__ slabF_c, int *__restrict__ slabB_j, double *__restrict__ slabB_c) {
    constexpr int NS = 2 * D;
    constexpr int TS = (NS + 1 <= 4) ? 4 : 8;  // FP32 tile row: centred position, velocity, v'Rv, padded to float4s
    constexpr bool FILL = (MODE == 1);
    constexpr int kRing = 128;  // >= 31 waiting + 64 pushed per step
    __shared__ __align__(16) float tile[kLqTile * TS];
    __shared__ double s_x[kLqThreads * NS];
    __shared__ unsigned s_ring[kLqThreads / 32][kRing];
    __shared__ int s_cnt[2][kLqThreads];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = w < nq;
    const int64_t q = q0 + w;
    // stage-1 operands of this thread's query in FP32: centred position, velocity, R v, v'Rv
    float xp[D], xv[D], Rxv[D], gx = 0.0f;
    {
        double x[NS];
#pragma unroll
        for (int i = 0; i < NS; ++i) {
            x[i] = active ? V[q * NS + i] : 0.0;
            s_x[threadIdx.x * NS + i] = x[i];
        }
#pragma unroll
        for (int i = 0; i < D; ++i) { xp[i] = (float)(x[i] - P.center[i]); xv[i] = (float)x[D + i]; }
#pragma unroll
        for (int i = 0; i < D; ++i) {
            float t = 0.0f;
#pragma unroll
            for (int j = 0; j < D; ++j) t = fmaf(P.R[i * D + j], xv[j], t);
            Rxv[i] = t;
            gx = fmaf(xv[i], t, gx);
        }
    }
    s_cnt[0][threadIdx.x] = 0;
    s_cnt[1][threadIdx.x] = 0;
    unsigned head = 0, tail = 0;  // warp-uniform ring positions (monotone; slot = pos % kRing)

    // stage 2 over the first n ring items (n <= 32); every lane of the warp calls it
    auto process = [&](int n) {
        const bool have = lane < n;
        const unsigned item = have ? s_ring[wid][(head + lane) % kRing] : 0u;
        const int owner = (int)(item >> 27), dir = (int)((item >> 26) & 1u);
        const int64_t j = (int64_t)(item & 0x3ffffffu);
        double c = 0.0;
        bool acc = false;
        if (have) {
            double from[NS], to[NS];  // forwards: owner -> sample; backwards: sample -> owner
#pragma unroll
            for (int i = 0; i < NS; ++i) {
                const double xo = s_x[(wid * 32 + owner) * NS + i], y = V[j * NS + i];
                from[i] = dir ? y : xo;
                to[i] = dir ? xo : y;
            }
            // the EXACT candidate test of the reference (cands = cd .> 0, linearquadratic.jl:213) decides here:
            // stage 1 only discarded pairs that provably fail it
            const Abg k = lq_abg<D>(L, from, to);
            if (lq_dcost(k, r) > 0) {
                if (same_state<D>(from, to)) c = 0.0;               // :192 (duplicate states)
                else c = lq_cost(k, lq_topt_newton(k, r));
                acc = c <= r;                                       // :221
            }
        }
        const unsigned peers = __match_any_sync(0xffffffffu, have ? (item >> 26) : (0x80000000u | (unsigned)lane));
        const unsigned accm = __ballot_sync(0xffffffffu, acc);
        const unsigned mine = peers & accm;
        if (acc) {
            const int col = wid * 32 + owner;
            const int slot = s_cnt[dir][col] + __popc(mine & ((1u << lane) - 1u));
            const int64_t wo = (int64_t)blockIdx.x * blockDim.x + col;
            if (FILL) {
                const int64_t pos = (dir ? colptrB[wo] : colptrF[wo]) - 1 + slot;
                if (dir) { rowvalB[pos] = j + 1; nzvalB[pos] = c; } else { rowvalF[pos] = j + 1; nzvalF[pos] = c; }
            }
            if (MODE == 2 && slot < cap) {
                if (dir) { slabB_j[wo * cap + slot] = (int)j; slabB_c[wo * cap + slot] = c; }
                else { slabF_j[wo * cap + slot] = (int)j; slabF_c[wo * cap + slot] = c; }
            }
        }
        __syncwarp();
        if (acc && (mine >> lane) == 1u)  // the last accepted item of this (owner, direction) in the batch
            s_cnt[dir][wid * 32 + owner] += __popc(mine);
        __syncwarp();
        head += (unsigned)n;
    };

    for (int64_t t0 = 0; t0 < N; t0 += kLqTile) {
        const int cnt = (int)((N - t0 < kLqTile) ? (N - t0) : kLqTile);
        __syncthreads();
        for (int jj = threadIdx.x; jj < cnt; jj += blockDim.x) {  // FP32 image of the tile (one sample per thread)
            float yv[D], g = 0.0f;
#pragma unroll
            for (int i = 0; i < D; ++i) {
                tile[jj * TS + i] = (float)(V[(t0 + jj) * NS + i] - P.center[i]);
                yv[i] = (float)V[(t0 + jj) * NS + D + i];
                tile[jj * TS + D + i] = yv[i];
            }
#pragma unroll
            for (int i = 0; i < D; ++i) {
                float t = 0.0f;
#pragma unroll
                for (int j2 = 0; j2 < D; ++j2) t = fmaf(P.R[i * D + j2], yv[j2], t);
                g = fmaf(yv[i], t, g);
            }
            tile[jj * TS + NS] = g;
        }
        __syncthreads();
        const int q_in_tile = (active && q >= t0 && q < t0 + cnt) ? (int)(q - t0) : -1;  // j == q as a 32-bit compare
        for (int jj = 0; jj < cnt; ++jj) {
            const int64_t j = t0 + jj;
            // stage 1, FP32 with FMA: dcost(r) = 1 - (36/r^4) dp'R dp - (4/r^2)(vx'Rvx + vx'Rvy + vy'Rvy) +- (24/r^3)(vx+vy)'R dp
            // (+ forwards x -> y, - backwards y -> x; gamma is symmetric for symmetric R).  A pair is kept when the
            // FP32 value exceeds -delta, delta bounding the FP32 evaluation error for this sample set (lq_prefilter):
            // a superset of cands = cd .> 0 (linearquadratic.jl:213); stage 2 applies the exact test.
            // j == q is dropped (nearneighbors.jl:171).
            const bool live = active && jj != q_in_tile;
            float row[TS];  // one or two 16-byte broadcast reads
#pragma unroll
            for (int v4 = 0; v4 < TS / 4; ++v4) {
                const float4 t4 = reinterpret_cast<const float4 *>(tile + jj * TS)[v4];
                row[4 * v4] = t4.x; row[4 * v4 + 1] = t4.y; row[4 * v4 + 2] = t4.z; row[4 * v4 + 3] = t4.w;
            }
            float dp[D], sv[D], a = 0.0f, b = 0.0f, g = gx + row[NS];
#pragma unroll
            for (int i = 0; i < D; ++i) {
                dp[i] = row[i] - xp[i];
                const float yvi = row[D + i];
                sv[i] = xv[i] + yvi;
                g = fmaf(Rxv[i], yvi, g);
            }
#pragma unroll
            for (int i = 0; i < D; ++i) {
                float t = 0.0f;
#pragma unroll
                for (int j2 = 0; j2 < D; ++j2) t = fmaf(P.R[i * D + j2], dp[j2], t);
                a = fmaf(dp[i], t, a);
                b = fmaf(sv[i], t, b);
            }
            const float base = fmaf(-P.c2, g, fmaf(-P.c4, a, 1.0f));
            // second necessary condition, the same for both directions: cost(t) = t + (alpha u^2 - beta u + gamma)/t with
            // u = 1/t >= t + D/t, D = gamma - beta^2/(4 alpha), so cost <= r needs 2 sqrt(D) <= r, i.e.
            // a (16 g - r^2) - 12 b^2 <= 0 (alpha = 12a, beta = +-12b, gamma = 4g).  98% of the dcost(r) > 0 candidates
            // fail it -- pairs whose optimum lies before r but costs more than r -- and never reach the Newton stage.
            const bool near = live && (fmaf(-12.0f * b, b, a * fmaf(16.0f, g, -P.r2)) <= P.delta2);
            const bool pf = near && (fmaf(P.c3, b, base) > P.neg_delta);
            const bool pb = near && (fmaf(-P.c3, b, base) > P.neg_delta);
            const unsigned mf = __ballot_sync(0xffffffffu, pf), mb = __ballot_sync(0xffffffffu, pb);
            if (mf | mb) {
                const unsigned lt = (1u << lane) - 1u;
                if (pf) s_ring[wid][(tail + __popc(mf & lt)) % kRing] = ((unsigned)lane << 27) | (unsigned)j;
                tail += __popc(mf);
                if (pb) s_ring[wid][(tail + __popc(mb & lt)) % kRing] = ((unsigned)lane << 27) | (1u << 26) | (unsigned)j;
                tail += __popc(mb);
                __syncwarp();
                while (tail - head >= 32u) process(32);
            }
        }
    }
    if (tail != head) process((int)(tail - head));  // < 32 left
    if (!FILL && active) { countsF[w] = s_cnt[0][threadIdx.x]; countsB[w] = s_cnt[1][threadIdx.x]; }
}

__global__ void __launch_bounds__(256)
lq_slab_to_csc(const int *__restrict__ slab_j, const double *__restrict__ slab_c, int cap, int64_t nq,
               const int64_t *__restrict__ colptr, int64_t *__restrict__ rowval, double *__restrict__ nzval) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t w = gw; w < nq; w += nw) {
        const int64_t base = colptr[w] - 1;
        const int k = (int)(colptr[w + 1] - colptr[w]);
        for (int e = lane; e < k; e += 32) {
            rowval[base + e] = (int64_t)slab_j[w * cap + e] + 1;
            nzval[base + e] = slab_c[w * cap + e];
        }
    }
}
__global__ void lq_max_count(const int *__restrict__ a, const int *__restrict__ b, int64_t n, int *__restrict__ out) {
    int m = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        m = max(m, max(a[i], b[i]));
    for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

template <int D>
__global__ void __launch_bounds__(256)
lq_steer_kernel(const double *__restrict__ A, const double *__restrict__ B, int64_t n, LqDev L, double r,
                double *__restrict__ cost, double *__restrict__ topt) {
    constexpr int NS = 2 * D;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double a[NS], b[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) { a[k] = A[i * NS + k]; b[k] = B[i * NS + k]; }
        double c, t;
        lq_steer<D>(L, a, b, r, &c, &t);
        cost[i] = c;
        topt[i] = t;
    }
}

// K9: is_free_motion(v, w, CC, SS) along the optimal trajectory; *checks += segment tests run
template <int D, int DW, int KIND>
__device__ __forceinline__ bool lq_motion_free(const LqDev &L, const SpaceDev &S, const double *T, int M, double r,
                                               const double *v, const double *w, int *checks) {
    constexpr int NS = 2 * D;
    double c, t;
    lq_steer<D>(L, v, w, r, &c, &t);
    double cur[NS], nxt[NS], p[DW], q[DW];
    lq_state<D>(v, w, t, 0.0, cur);
    state2workspace<NS, DW>(S, cur, p);
    for (int i = 1; i <= 4; ++i) {
        if (!in_state_space<NS>(S, cur)) return false;  // only wps[1..4] are bounds-checked (Q4)
        const double s = ddiv(dmul((double)i, t), 4.0);  // linspace(0, t, 5)[i+1]
        lq_state<D>(v, w, t, s, nxt);
        state2workspace<NS, DW>(S, nxt, q);
        *checks += 1;
        bool free_;
        if (KIND == 0) free_ = !line_colliding_2d(T, p[0], p[DW > 1 ? 1 : 0], q[0], q[DW > 1 ? 1 : 0]);
        else free_ = box_segment_free<DW>(T, M, p, q);
        if (!free_) return false;
#pragma unroll
        for (int k = 0; k < NS; ++k) cur[k] = nxt[k];
#pragma unroll
        for (int k = 0; k < DW; ++k) p[k] = q[k];
    }
    return true;
}

__device__ __forceinline__ const double *lq_stage_table(const double *__restrict__ g_table, int words, bool use_smem,
                                                        double *smem) {
    if (!use_smem) return g_table;
    for (int i = threadIdx.x; i < words; i += blockDim.x) smem[i] = g_table[i];
    __syncthreads();
    return smem;
}

// one warp per column of the (backwards) table: entry (row y -> column x) = motion V[y] -> V[x]
template <int D, int DW, int KIND>
__global__ void __launch_bounds__(256)
lq_edges_free_kernel(const double *__restrict__ V, const int64_t *__restrict__ colptr,
                     const int64_t *__restrict__ rowval, int64_t ncols, int64_t col0, LqDev L, double r, SpaceDev S,
                     const double *__restrict__ g_table, int table_words, int M, bool use_smem,
                     uint32_t *__restrict__ bits32, unsigned long long *__restrict__ checks) {
    constexpr int NS = 2 * D;
    extern __shared__ double s_table[];
    const double *T = lq_stage_table(g_table, table_words, use_smem, s_table);
    const int lane = threadIdx.x & 31;
    const int64_t gwarp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    unsigned long long my_checks = 0;
    for (int64_t c = gwarp; c < ncols; c += nwarps) {
        const int64_t beg = colptr[c] - 1, end = colptr[c + 1] - 1;
        if (beg >= end) continue;
        double b[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) b[k] = V[(col0 + c) * NS + k];
        for (int64_t e0 = beg; e0 < end; e0 += 32) {
            const int64_t e = e0 + lane;
            bool ok = false;
            if (e < end) {
                const int64_t y = rowval[e] - 1;
                double a[NS];
#pragma unroll
                for (int k = 0; k < NS; ++k) a[k] = V[y * NS + k];
                int nchk = 0;
                ok = lq_motion_free<D, DW, KIND>(L, S, T, M, r, a, b, &nchk);
                my_checks += nchk;
            }
            const unsigned m = __ballot_sync(0xffffffffu, ok);
            if (lane == 0 && m) {
                const int sh = (int)(e0 & 31);
                const int64_t wi = e0 >> 5;
                atomicOr(&bits32[wi], m << sh);
                if (sh && (m >> (32 - sh))) atomicOr(&bits32[wi + 1], m >> (32 - sh));
            }
        }
    }
    __shared__ unsigned long long s_checks[8];
#pragma unroll
    for (int o = 16; o; o >>= 1) my_checks += __shfl_xor_sync(0xffffffffu, my_checks, o);
    if (lane == 0) s_checks[threadIdx.x >> 5] = my_checks;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < 8; ++w) t += s_checks[w];
        if (t) atomicAdd(checks, t);
    }
}

template <int D, int DW, int KIND>
__global__ void __launch_bounds__(256)
lq_motions_free_kernel(const double *__restrict__ A, const double *__restrict__ B, int64_t n, LqDev L, double r,
                       SpaceDev S, const double *__restrict__ g_table, int table_words, int M, bool use_smem,
                       uint8_t *__restrict__ out, unsigned long long *__restrict__ checks) {
    constexpr int NS = 2 * D;
    extern __shared__ double s_table[];
    const double *T = lq_stage_table(g_table, table_words, use_smem, s_table);
    unsigned long long my_checks = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double a[NS], b[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) { a[k] = A[i * NS + k]; b[k] = B[i * NS + k]; }
        int nchk = 0;
        out[i] = lq_motion_free<D, DW, KIND>(L, S, T, M, r, a, b, &nchk) ? 1 : 0;
        my_checks += nchk;
    }
    if (my_checks) atomicAdd(checks, my_checks);
}

// ---- host side ---------------------------------------------------------------------------------
int make_space(const mpb200_space_desc *ss, int d_state, SpaceDev *out, int *dw);

static LqDev lq_dev(const mpb200_lq *lq) {
    LqDev L;
    L.scalar_R = lq->scalar_R ? 1 : 0;
    for (int i = 0; i < 9; ++i) L.R[i] = lq->R[i];
    return L;
}

// Stage 1 evaluates  dcost(r) = 1 - c4 a - c2 g +- c3 b  in FP32 (a = dp'R dp, b = (vx+vy)'R dp, g = vx'Rvx + vx'Rvy +
// vy'Rvy) from FP32-rounded inputs.  Standard forward error bound for sums of products: |fl(e) - e| <= gamma_k * (sum of
// the absolute values of the terms), gamma_k = k u / (1 - k u), u = 2^-24; every term is a product of <= 3 rounded inputs
// reached through <= 12 roundings, so k = 24 covers it; the term magnitudes are bounded with the sample set's own
// extents (centred positions |p| <= Mp, velocities |v| <= Mv, rho = max row sum of |R|):
//   a <= rho D (2Mp)^2,  |b| <= rho D (2Mv)(2Mp),  g <= 3 rho D Mv^2.
// delta = 2 * gamma_24 * (1 + c4 a_max + c3 b_max + c2 g_max): twice the bound, so no pair with exact dcost(r) > 0 is lost.
template <int D>
static LqPre lq_prefilter(const mpb200_samples *s, const mpb200_lq *lq, double r) {
    LqPre P;
    memset(&P, 0, sizeof(P));
    double Mp = 0, Mv = 0, rho = 0;
    for (int i = 0; i < D; ++i) {
        P.center[i] = 0.5 * (s->h_bbox[i] + s->h_bbox[2 * D + i]);
        Mp = fmax(Mp, fmax(fabs(s->h_bbox[i] - P.center[i]), fabs(s->h_bbox[2 * D + i] - P.center[i])));
        Mv = fmax(Mv, fmax(fabs(s->h_bbox[D + i]), fabs(s->h_bbox[2 * D + D + i])));
        double row = 0;
        for (int j = 0; j < D; ++j) { P.R[i * D + j] = (float)lq->R[i * D + j]; row += fabs(lq->R[i * D + j]); }
        rho = fmax(rho, row);
    }
    const double c2 = 4.0 / (r * r), c3 = 24.0 / (r * r * r), c4 = 36.0 / (r * r * r * r);
    P.c2 = (float)c2; P.c3 = (float)c3; P.c4 = (float)c4;
    const double u = 5.9604644775390625e-08, gk = 24.0 * u / (1.0 - 24.0 * u);
    const double S = 1.0 + c4 * rho * D * 4.0 * Mp * Mp + c3 * rho * D * 4.0 * Mv * Mp + c2 * 3.0 * rho * D * Mv * Mv;
    double delta = 2.0 * gk * S;
    if (!(delta < 1e30)) delta = 1e30;  // absurd extents: the prefilter keeps everything, stage 2 still decides exactly
    P.neg_delta = -(float)delta;
    P.neg_delta = nextafterf(P.neg_delta, -INFINITY);
    // w = a (16 g - r^2) - 12 b^2: same error model, 16 roundings deep; twice the bound again.  A pair is dropped only
    // if w > delta2, i.e. exactly 4 D - r^2 = w / a >= delta2 / (2 a_max) > 0: its cost exceeds r by a margin many
    // orders above the FP64 rounding of the reference's own cost evaluation.
    const double am = rho * D * 4.0 * Mp * Mp, bm = rho * D * 4.0 * Mv * Mp, gm = 3.0 * rho * D * Mv * Mv;
    const double g16 = 16.0 * u / (1.0 - 16.0 * u);
    double d2 = 2.0 * g16 * (am * (16.0 * gm + r * r) + 12.0 * bm * bm);
    if (!(d2 < 1e30)) d2 = 1e30;
    P.r2 = (float)(r * r);
    P.delta2 = nextafterf((float)d2, INFINITY);
    return P;
}

template <int D>
static int lq_build(mpb200_samples *s, const mpb200_lq *lq, double r, mpb200_table *tF, mpb200_table *tB) {
    Context &c = ctx();
    cudaStream_t st = c.stream;
    const int64_t N = s->N, nq = s->q1 - s->q0;
    const double *V = s->V.as<double>();
    const LqDev L = lq_dev(lq);
    const LqPre P = lq_prefilter<D>(s, lq, r);
    for (mpb200_table *t : {tF, tB}) {
        if (int rc = t->counts.reserve(sizeof(int) * (size_t)(nq + 1))) return rc;
        if (int rc = t->colptr.reserve(sizeof(int64_t) * (size_t)(nq + 1))) return rc;
    }
    const unsigned nb = (unsigned)ceil_div(nq > 0 ? nq : 1, kLqThreads);
    int *d_max = reinterpret_cast<int *>(c.d_scalar + 2);
    phase_bank(MPB200_OP_TABLE);
    phase_mark(0);
    // slab capacity from a probe of up to 1024 query columns (exact counts for those columns)
    int cap = 0;
    if (nq > 0) {
        const int64_t probe = nq < 1024 ? nq : 1024;
        MPB_CUDA(cudaMemsetAsync(d_max, 0, sizeof(int), st));
        lq_inball_kernel<D, 0><<<(unsigned)ceil_div(probe, kLqThreads), kLqThreads, 0, st>>>(
            V, N, s->q0, probe, L, P, r, tF->counts.as<int>(), tB->counts.as<int>(), nullptr, nullptr, nullptr, nullptr,
            nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr);
        MPB_LAUNCHED();
        lq_max_count<<<8, 256, 0, st>>>(tF->counts.as<int>(), tB->counts.as<int>(), probe, d_max);
        MPB_LAUNCHED();
        int h_max = 0;
        MPB_CUDA(cudaMemcpyAsync(&h_max, d_max, sizeof(int), cudaMemcpyDeviceToHost, st));
        MPB_CUDA(cudaStreamSynchronize(st));
        cap = (probe == nq) ? h_max : (2 * h_max + 64);
        cap = (cap + 31) & ~31;
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        if (cap == 0 || 56.0 * (double)cap * (double)nq > 0.8 * (double)free_b) cap = 0;
    }
    bool single = cap > 0;
    int *slabF_j = nullptr, *slabB_j = nullptr;
    double *slabF_c = nullptr, *slabB_c = nullptr;
    if (single) {
        const size_t per = (size_t)cap * (size_t)nq;
        if (int rc = tF->scratch.reserve(24 * per + 64)) return rc;
        slabF_c = tF->scratch.as<double>();
        slabB_c = slabF_c + per;
        slabF_j = reinterpret_cast<int *>(slabB_c + per);
        slabB_j = slabF_j + per;
    }
    if (nq > 0) {
        if (single) {
            lq_inball_kernel<D, 2><<<nb, kLqThreads, 0, st>>>(V, N, s->q0, nq, L, P, r, tF->counts.as<int>(),
                                                             tB->counts.as<int>(), nullptr, nullptr, nullptr, nullptr,
                                                             nullptr, nullptr, cap, slabF_j, slabF_c, slabB_j, slabB_c);
            MPB_LAUNCHED();
            MPB_CUDA(cudaMemsetAsync(d_max, 0, sizeof(int), st));
            lq_max_count<<<64, 256, 0, st>>>(tF->counts.as<int>(), tB->counts.as<int>(), nq, d_max);
        } else {
            lq_inball_kernel<D, 0><<<nb, kLqThreads, 0, st>>>(V, N, s->q0, nq, L, P, r, tF->counts.as<int>(),
                                                             tB->counts.as<int>(), nullptr, nullptr, nullptr, nullptr,
                                                             nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr);
        }
        MPB_LAUNCHED();
    }
    if (int rc = exclusive_scan<int, int64_t>(tF->counts.as<int>(), nq, tF->colptr.as<int64_t>(), (int64_t)1, s->scan_tmp,
                                              c.d_scalar))
        return rc;
    if (int rc = exclusive_scan<int, int64_t>(tB->counts.as<int>(), nq, tB->colptr.as<int64_t>(), (int64_t)1, s->scan_tmp,
                                              c.d_scalar + 1))
        return rc;
    phase_mark(1);
    MPB_CUDA(cudaMemcpyAsync(c.h_scalar, c.d_scalar, sizeof(int64_t) * 3, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    const int64_t nnzF = c.h_scalar[0], nnzB = c.h_scalar[1];
    if (single && *reinterpret_cast<int *>(c.h_scalar + 2) > cap) single = false;  // a slab overflowed
    if (int rc = tF->rowval.reserve(sizeof(int64_t) * (size_t)(nnzF + 1))) return rc;
    if (int rc = tF->nzval.reserve(sizeof(double) * (size_t)(nnzF + 1))) return rc;
    if (int rc = tB->rowval.reserve(sizeof(int64_t) * (size_t)(nnzB + 1))) return rc;
    if (int rc = tB->nzval.reserve(sizeof(double) * (size_t)(nnzB + 1))) return rc;
    phase_mark(2);
    if (nq > 0 && (nnzF > 0 || nnzB > 0)) {
        if (single) {
            const unsigned g2 = (unsigned)(ctx().sm_count * 8);
            lq_slab_to_csc<<<g2, 256, 0, st>>>(slabF_j, slabF_c, cap, nq, tF->colptr.as<int64_t>(), tF->rowval.as<int64_t>(),
                                               tF->nzval.as<double>());
            MPB_LAUNCHED();
            lq_slab_to_csc<<<g2, 256, 0, st>>>(slabB_j, slabB_c, cap, nq, tB->colptr.as<int64_t>(), tB->rowval.as<int64_t>(),
                                               tB->nzval.as<double>());
        } else {
            lq_inball_kernel<D, 1><<<nb, kLqThreads, 0, st>>>(V, N, s->q0, nq, L, P, r, nullptr, nullptr,
                                                             tF->colptr.as<int64_t>(), tB->colptr.as<int64_t>(),
                                                             tF->rowval.as<int64_t>(), tF->nzval.as<double>(),
                                                             tB->rowval.as<int64_t>(), tB->nzval.as<double>(), 0, nullptr,
                                                             nullptr, nullptr, nullptr);
        }
        MPB_LAUNCHED();
    }
    phase_mark(3);
    MPB_CUDA(cudaStreamSynchronize(st));
    phases_collect(3);
    tF->ncols = tB->ncols = nq;
    tF->col0 = tB->col0 = s->q0;
    tF->nnz = nnzF;
    tB->nnz = nnzB;
    tF->r = tB->r = r;
    tF->euclid = tB->euclid = false;
    tF->has_order = tB->has_order = false;
    return 0;
}

int lq_inball_build(mpb200_samples *s, const mpb200_lq *lq, double r, mpb200_table *tF, mpb200_table *tB) {
    if (s->N >= (int64_t(1) << 26)) return fail(MPB200_EARG, "all-pairs LQ tables support N < 2^26 samples");
    if (s->d != 2 * lq->d) return fail(MPB200_EARG, "sample dimension %d != 2 x %d", s->d, lq->d);
    if (lq->d == 1) return lq_build<1>(s, lq, r, tF, tB);
    if (lq->d == 2) return lq_build<2>(s, lq, r, tF, tB);
    if (lq->d == 3) return lq_build<3>(s, lq, r, tF, tB);
    return fail(MPB200_EARG, "double integrators of dimension 1..3 are built in (got %d)", lq->d);
}

int lq_steer_device(const mpb200_lq *lq, const double *dA, const double *dB, int64_t n, double r, double *d_cost,
                    double *d_topt) {
    const LqDev L = lq_dev(lq);
    cudaStream_t st = ctx().stream;
    const unsigned grid = (unsigned)(ceil_div(n, 256) < 148 * 8 ? ceil_div(n, 256) : 148 * 8);
    if (lq->d == 1) lq_steer_kernel<1><<<grid, 256, 0, st>>>(dA, dB, n, L, r, d_cost, d_topt);
    else if (lq->d == 2) lq_steer_kernel<2><<<grid, 256, 0, st>>>(dA, dB, n, L, r, d_cost, d_topt);
    else if (lq->d == 3) lq_steer_kernel<3><<<grid, 256, 0, st>>>(dA, dB, n, L, r, d_cost, d_topt);
    else return fail(MPB200_EARG, "double integrators of dimension 1..3 are built in (got %d)", lq->d);
    MPB_LAUNCHED();
    return 0;
}

struct LqLaunch {
    const double *table;
    int words, M;
    bool use_smem;
    size_t smem;
};
static LqLaunch lq_cfg(const mpb200_obstacles *o) {
    LqLaunch C;
    C.table = o->table.as<double>();
    C.words = o->table_words;
    C.M = o->M;
    size_t bytes = sizeof(double) * (size_t)o->table_words;
    C.use_smem = bytes <= 160 * 1024;
    C.smem = C.use_smem ? bytes : 0;
    return C;
}

// (D, DW, KIND) combinations: workspace = positions of the double integrator
#define MPB_LQ_DISPATCH(D_, DW_, KIND_, CALL)                                                       \
    do {                                                                                            \
        if (KIND_ == 0 && DW_ != 2) return fail(MPB200_EARG, "2-D obstacles need a 2-D workspace"); \
        if (D_ == 2 && DW_ == 2 && KIND_ == 0) { CALL(2, 2, 0); }                                   \
        else if (D_ == 2 && DW_ == 2 && KIND_ == 1) { CALL(2, 2, 1); }                              \
        else if (D_ == 3 && DW_ == 3 && KIND_ == 1) { CALL(3, 3, 1); }                              \
        else if (D_ == 3 && DW_ == 2 && KIND_ == 0) { CALL(3, 2, 0); }                              \
        else if (D_ == 1 && DW_ == 1 && KIND_ == 1) { CALL(1, 1, 1); }                              \
        else return fail(MPB200_EARG, "unsupported LQ (d=%d, workspace=%d, checker=%d) combination", D_, DW_, KIND_); \
    } while (0)

int lq_edges_free_device(const mpb200_samples *s, const mpb200_table *t, const mpb200_lq *lq, double r,
                         const mpb200_obstacles *o, const mpb200_space_desc *ss, uint32_t *d_bits32,
                         unsigned long long *d_checks) {
    SpaceDev S;
    int dw = 0;
    if (int rc = make_space(ss, s->d, &S, &dw)) return rc;
    if (s->d != 2 * lq->d) return fail(MPB200_EARG, "sample dimension %d != 2 x %d", s->d, lq->d);
    if (o->kind == 1 && o->d != dw) return fail(MPB200_EARG, "box dimension %d != workspace dimension %d", o->d, dw);
    const LqDev L = lq_dev(lq);
    const LqLaunch C = lq_cfg(o);
    cudaStream_t st = ctx().stream;
    int64_t blocks = ceil_div(t->ncols > 0 ? t->ncols : 1, 8);
    const unsigned grid = (unsigned)(blocks < (int64_t)ctx().sm_count * 8 ? blocks : (int64_t)ctx().sm_count * 8);
#define CALL(D_, DW_, K_)                                                                                          \
    do {                                                                                                           \
        if (C.smem > 48 * 1024)                                                                                    \
            MPB_CUDA(cudaFuncSetAttribute(lq_edges_free_kernel<D_, DW_, K_>,                                       \
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C.smem));              \
        lq_edges_free_kernel<D_, DW_, K_><<<grid, 256, C.smem, st>>>(                                              \
            s->V.as<double>(), t->colptr.as<int64_t>(), t->rowval.as<int64_t>(), t->ncols, t->col0, L, r, S, C.table, \
            C.words, C.M, C.use_smem, d_bits32, d_checks);                                                         \
    } while (0)
    MPB_LQ_DISPATCH(lq->d, dw, o->kind, CALL);
#undef CALL
    MPB_LAUNCHED();
    return 0;
}

int lq_motions_free_device(const mpb200_lq *lq, double r, const double *dA, const double *dB, int64_t n, int d_state,
                           const mpb200_obstacles *o, const mpb200_space_desc *ss, uint8_t *d_out,
                           unsigned long long *d_checks) {
    SpaceDev S;
    int dw = 0;
    if (int rc = make_space(ss, d_state, &S, &dw)) return rc;
    if (d_state != 2 * lq->d) return fail(MPB200_EARG, "state dimension %d != 2 x %d", d_state, lq->d);
    if (o->kind == 1 && o->d != dw) return fail(MPB200_EARG, "box dimension %d != workspace dimension %d", o->d, dw);
    const LqDev L = lq_dev(lq);
    const LqLaunch C = lq_cfg(o);
    cudaStream_t st = ctx().stream;
    const unsigned grid = (unsigned)(ceil_div(n, 256) < 148 * 8 ? ceil_div(n, 256) : 148 * 8);
#define CALL(D_, DW_, K_)                                                                                       \
    do {                                                                                                        \
        if (C.smem > 48 * 1024)                                                                                 \
            MPB_CUDA(cudaFuncSetAttribute(lq_motions_free_kernel<D_, DW_, K_>,                                  \
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C.smem));           \
        lq_motions_free_kernel<D_, DW_, K_><<<grid, 256, C.smem, st>>>(dA, dB, n, L, r, S, C.table, C.words, C.M, \
                                                                       C.use_smem, d_out, d_checks);            \
    } while (0)
    MPB_LQ_DISPATCH(lq->d, dw, o->kind, CALL);
#undef CALL
    MPB_LAUNCHED();
    return 0;
}

// lazy GMT*: step 4 runs lq_motion_free (the check of lq_edges_free_kernel) on the winning entry, on one lane
template <int D, int DW, int KIND>
struct GmtLqEdge {
    static constexpr bool kLazy = true;
    LqDev L;
    double r;
    SpaceDev S;
    const double *T;
    int M;
    __device__ bool operator()(const GmtArgs &a, long long, int y, int x, GmtCtl *ctl) const {
        double v[2 * D], w[2 * D];
        gmt_endpoints<2 * D>(a, y, x, v, w);
        int nchk = 0;
        const bool ok = lq_motion_free<D, DW, KIND>(L, S, T, M, r, v, w, &nchk);
        gmt_count_segments(ctl, nchk);
        return ok;
    }
};

int gmt_lazy_lq(const GmtArgs &a, const mpb200_lq *lq, double r, const mpb200_obstacles *o, const mpb200_space_desc *ss,
                int *blocks) {
    SpaceDev S;
    int dw = 0;
    if (int rc = make_space(ss, a.d, &S, &dw)) return rc;
    if (a.d != 2 * lq->d) return fail(MPB200_EARG, "sample dimension %d != 2 x %d", a.d, lq->d);
    if (o->kind == 1 && o->d != dw) return fail(MPB200_EARG, "box dimension %d != workspace dimension %d", o->d, dw);
    const LqDev L = lq_dev(lq);
#define CALL(D_, DW_, K_) return gmt_launch(a, GmtLqEdge<D_, DW_, K_>{L, r, S, o->table.as<double>(), o->M}, blocks)
    MPB_LQ_DISPATCH(lq->d, dw, o->kind, CALL);
#undef CALL
    return 0;
}

}  // namespace mpb
