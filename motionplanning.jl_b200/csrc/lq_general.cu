// lq_general.cu -- K5 / K9 for GENERAL linear-affine systems  xdot = A x + B u + c  (nilpotent A, drift c).
//
// Replaces LinearQuadratic(A, B, c, R) / LinearQuadratic2BVP (linearquadratic.jl:28-39, 94-157) beyond the
// double-integrator closed form of lq.cu: where the reference prints SymPy expressions into closures, this
// evaluates the same quantities numerically from per-system tables
//     Ak = A^k / k!,  dk = Ak c / (k+1),  BRB = B R^-1 B',  G(t) = sum_p Gp t^p
// per (x, y, t):  xbar = e^{At} x + int e^{As} c,  e = y - xbar,  lam = G^-1 e  (Cholesky),
//     cost = t + e'lam,   dcost = 1 - 2 lam'(A y + c) - lam' BRB lam,   ddcost = 2 (mu + A'lam)'h,
//     h = A y + c + BRB lam,  mu = G^-1 h;      x(s) = xbar(s) + G(s) e^{A'(t-s)} lam(t)
// (dcost at t = r is the reference's dense prefilter, linearquadratic.jl:205-211).  The operation order is the
// one specified in oracle/lq_general.c, every operation an explicit _rn intrinsic, so tables, costs and validity
// bits are bit-identical to the oracle; the oracle itself is pinned to the reference's SymPy construction by
// tests/golden/lq_general.json.  steer / topt_newton: linearquadratic.jl:160-195; tables: :68-77,196-225 +
// nearneighbors.jl:165-177; waypoints: :85-88 with statespaces.jl:153-158.
//
// Layout: the tables (a few KB) are staged in shared memory once per CTA; one thread per query column walks the
// samples (tiles through shared memory, broadcast reads) in index order, both directions, so rows come out
// ascending; count pass + fill pass.  This is the general path: the double-integrator family keeps lq.cu's
// closed form and its two-stage survivor pipeline.
#include "common.cuh"
#include "predicates.cuh"
#include "scan.cuh"
#include "lq_general.cuh"
#include <cmath>

namespace mpb {

// ---- host: tables (same procedure, same operation order as oracle/lq_general.c: orc_lqg_setup) -------------
static void h_matmul(int n, const double *X, const double *Y, double *Z) {
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            double s = 0;
            for (int k = 0; k < n; ++k) s = s + X[i * n + k] * Y[k * n + j];
            Z[i * n + j] = s;
        }
}
static bool h_chol(int n, const double *G, double *Lw) {
    for (int i = 0; i < n; ++i)
        for (int j = 0; j <= i; ++j) {
            double s = G[i * n + j];
            for (int k = 0; k < j; ++k) s = s - Lw[i * n + k] * Lw[j * n + k];
            if (i == j) {
                if (!(s > 0)) return false;
                Lw[i * n + i] = sqrt(s);
            } else {
                Lw[i * n + j] = s / Lw[j * n + j];
            }
        }
    return true;
}
static void h_chol_solve(int n, const double *Lw, const double *b, double *x) {
    double y[kLqgMaxN];
    for (int i = 0; i < n; ++i) {
        double s = b[i];
        for (int k = 0; k < i; ++k) s = s - Lw[i * n + k] * y[k];
        y[i] = s / Lw[i * n + i];
    }
    for (int i = n - 1; i >= 0; --i) {
        double s = y[i];
        for (int k = i + 1; k < n; ++k) s = s - Lw[k * n + i] * x[k];
        x[i] = s / Lw[i * n + i];
    }
}

// A, B, R row-major here.  Returns MPB200_OK or MPB200_EARG with the message set.
int lqg_setup_host(int n, int m, const double *A, const double *B, const double *c, const double *R, LqgHost *S) {
    constexpr int GN = kLqgMaxN;
    if (n < 1 || n > GN || m < 1 || m > GN) return fail(MPB200_EARG, "general LQ systems support 1 <= n, m <= %d", GN);
    memset(S, 0, sizeof(*S));
    S->n = n;
    for (int i = 0; i < n * n; ++i) S->A[i] = A[i];
    for (int i = 0; i < n; ++i) S->c[i] = c[i];
    double P[GN * GN], Q[GN * GN];
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) P[i * n + j] = (i == j) ? 1.0 : 0.0;
    double fact = 1.0;
    for (int k = 0; k < n; ++k) {
        if (k > 0) { h_matmul(n, P, A, Q); memcpy(P, Q, sizeof(double) * n * n); fact = fact * (double)k; }
        for (int i = 0; i < n * n; ++i) S->Ak[k][i] = P[i] / fact;
    }
    h_matmul(n, P, A, Q);
    for (int i = 0; i < n * n; ++i)
        if (Q[i] != 0.0)  // linearquadratic.jl:96
            return fail(MPB200_EARG, "TODO: implement more cases than nilpotent A! (e.g. diagonalizable)");
    for (int k = 0; k < n; ++k)
        for (int i = 0; i < n; ++i) {
            double s = 0;
            for (int j = 0; j < n; ++j) s = s + S->Ak[k][i * n + j] * c[j];
            S->dk[k][i] = s / (double)(k + 1);
        }
    double Lr[GN * GN], Rinv[GN * GN], ej[GN], col[GN];
    if (!h_chol(m, R, Lr)) return fail(MPB200_EARG, "R must be symmetric positive definite");
    for (int j = 0; j < m; ++j) {
        for (int i = 0; i < m; ++i) ej[i] = (i == j) ? 1.0 : 0.0;
        h_chol_solve(m, Lr, ej, col);
        for (int i = 0; i < m; ++i) Rinv[i * m + j] = col[i];
    }
    double BR[GN * GN];
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < m; ++j) {
            double s = 0;
            for (int k = 0; k < m; ++k) s = s + B[i * m + k] * Rinv[k * m + j];
            BR[i * m + j] = s;
        }
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            double s = 0;
            for (int k = 0; k < m; ++k) s = s + BR[i * m + k] * B[j * m + k];
            S->BRB[i * n + j] = s;
        }
    S->np = 2 * n - 1;
    for (int p = 1; p <= S->np; ++p) {
        double acc[GN * GN];
        for (int i = 0; i < n * n; ++i) acc[i] = 0;
        for (int i = 0; i < n; ++i) {
            const int j = p - 1 - i;
            if (j < 0 || j >= n) continue;
            double T1[GN * GN];
            h_matmul(n, S->Ak[i], S->BRB, T1);
            for (int a = 0; a < n; ++a)
                for (int b = 0; b < n; ++b) {
                    double s = 0;
                    for (int k = 0; k < n; ++k) s = s + T1[a * n + k] * S->Ak[j][b * n + k];
                    acc[a * n + b] = acc[a * n + b] + s;
                }
        }
        for (int i = 0; i < n * n; ++i) S->Gp[p - 1][i] = acc[i] / (double)p;
    }
    // G(1) must be positive definite: the pair (A, B) is controllable (otherwise no finite steering cost exists)
    double G1[GN * GN], L1[GN * GN];
    for (int i = 0; i < n * n; ++i) {
        G1[i] = 0;
        for (int p = 0; p < S->np; ++p) G1[i] += S->Gp[p][i];
    }
    if (!h_chol(n, G1, L1)) return fail(MPB200_EARG, "(A, B) is not controllable: the Gramian is singular");
    return MPB200_OK;
}

template <int NS>
static void lqg_pack(const LqgHost &H, LqgTab<NS> *T) {
    memset(T, 0, sizeof(*T));
    for (int i = 0; i < NS * NS; ++i) { T->A[i] = H.A[i]; T->BRB[i] = H.BRB[i]; }
    for (int i = 0; i < NS; ++i) T->c[i] = H.c[i];
    for (int k = 0; k < NS; ++k) {
        for (int i = 0; i < NS * NS; ++i) T->Ak[k][i] = H.Ak[k][i];
        for (int i = 0; i < NS; ++i) T->dk[k][i] = H.dk[k][i];
    }
    for (int p = 0; p < 2 * NS - 1; ++p)
        for (int i = 0; i < NS * NS; ++i) T->Gp[p][i] = H.Gp[p][i];
}

template <int NS, bool FILL>
__global__ void __launch_bounds__(kLqgThreads)
lqg_inball_kernel(const double *__restrict__ V, int64_t N, int64_t q0, int64_t nq, const LqgTab<NS> *__restrict__ g_tab,
                  double r, int *__restrict__ countsF, int *__restrict__ countsB, const int64_t *__restrict__ colptrF,
                  const int64_t *__restrict__ colptrB, int64_t *__restrict__ rowvalF, double *__restrict__ nzvalF,
                  int64_t *__restrict__ rowvalB, double *__restrict__ nzvalB) {
    __shared__ LqgTab<NS> s_tab;
    __shared__ double tile[kLqgTile * NS];
    const LqgTab<NS> &S = lqg_stage<NS>(g_tab, &s_tab);
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = w < nq;
    const int64_t q = q0 + w;
    double x[NS];
#pragma unroll
    for (int i = 0; i < NS; ++i) x[i] = active ? V[q * NS + i] : 0.0;
    int cF = 0, cB = 0;
    int64_t pF = (FILL && active) ? colptrF[w] - 1 : 0, pB = (FILL && active) ? colptrB[w] - 1 : 0;
    for (int64_t t0 = 0; t0 < N; t0 += kLqgTile) {
        const int cnt = (int)((N - t0 < kLqgTile) ? (N - t0) : kLqgTile);
        __syncthreads();
        for (int i = threadIdx.x; i < cnt * NS; i += blockDim.x) tile[i] = V[t0 * NS + i];
        __syncthreads();
        if (!active) continue;
        for (int jj = 0; jj < cnt; ++jj) {
            const int64_t j = t0 + jj;
            if (j == q) continue;  // nearneighbors.jl:171
            double y[NS];
#pragma unroll
            for (int i = 0; i < NS; ++i) y[i] = tile[jj * NS + i];
#pragma unroll 1
            for (int dir = 0; dir < 2; ++dir) {  // 0: x -> y (forward table), 1: y -> x (backward table)
                const double *from = dir ? y : x, *to = dir ? x : y;
                if (!(lqg_dcost<NS>(S, from, to, r) > 0)) continue;  // cands = cd .> 0, linearquadratic.jl:213
                double c, t;
                lqg_steer<NS>(S, from, to, r, &c, &t);
                if (c <= r) {                                        // :221
                    if (dir == 0) {
                        if (FILL) { rowvalF[pF] = j + 1; nzvalF[pF] = c; ++pF; }
                        ++cF;
                    } else {
                        if (FILL) { rowvalB[pB] = j + 1; nzvalB[pB] = c; ++pB; }
                        ++cB;
                    }
                }
            }
        }
    }
    if (!FILL && active) { countsF[w] = cF; countsB[w] = cB; }
}

template <int NS>
__global__ void __launch_bounds__(128)
lqg_steer_kernel(const double *__restrict__ A, const double *__restrict__ B, int64_t n, const LqgTab<NS> *__restrict__ g_tab,
                 double r, double *__restrict__ cost, double *__restrict__ topt) {
    __shared__ LqgTab<NS> s_tab;
    const LqgTab<NS> &S = lqg_stage<NS>(g_tab, &s_tab);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double a[NS], b[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) { a[k] = A[i * NS + k]; b[k] = B[i * NS + k]; }
        double c, t;
        lqg_steer<NS>(S, a, b, r, &c, &t);
        cost[i] = c;
        topt[i] = t;
    }
}

// lane per stored entry (row y -> column x) = motion V[y] -> V[x]; edges taken in storage order
template <int NS, int DW, int KIND>
__global__ void __launch_bounds__(128)
lqg_edges_free_kernel(const double *__restrict__ V, const int64_t *__restrict__ colptr, const int64_t *__restrict__ rowval,
                      int64_t ncols, int64_t col0, const LqgTab<NS> *__restrict__ g_tab, double r, SpaceDev S,
                      const double *__restrict__ g_table, int table_words, int M, uint32_t *__restrict__ bits32,
                      unsigned long long *__restrict__ checks) {
    __shared__ LqgTab<NS> s_tab;
    const LqgTab<NS> &L = lqg_stage<NS>(g_tab, &s_tab);
    const double *T = g_table;  // the obstacle table is read through L1 here (the system tables own the shared memory)
    (void)table_words;
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
                ok = lqg_motion_free<NS, DW, KIND>(L, S, T, M, r, a, b, &nchk);
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
#pragma unroll
    for (int o = 16; o; o >>= 1) my_checks += __shfl_xor_sync(0xffffffffu, my_checks, o);
    if (lane == 0 && my_checks) atomicAdd(checks, my_checks);
}

template <int NS, int DW, int KIND>
__global__ void __launch_bounds__(128)
lqg_motions_free_kernel(const double *__restrict__ A, const double *__restrict__ B, int64_t n,
                        const LqgTab<NS> *__restrict__ g_tab, double r, SpaceDev S, const double *__restrict__ g_table,
                        int M, uint8_t *__restrict__ out, unsigned long long *__restrict__ checks) {
    __shared__ LqgTab<NS> s_tab;
    const LqgTab<NS> &L = lqg_stage<NS>(g_tab, &s_tab);
    unsigned long long my_checks = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double a[NS], b[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) { a[k] = A[i * NS + k]; b[k] = B[i * NS + k]; }
        int nchk = 0;
        out[i] = lqg_motion_free<NS, DW, KIND>(L, S, g_table, M, r, a, b, &nchk) ? 1 : 0;
        my_checks += nchk;
    }
    if (my_checks) atomicAdd(checks, my_checks);
}

// ---- host side ------------------------------------------------------------------------------------------
int make_space(const mpb200_space_desc *ss, int d_state, SpaceDev *out, int *dw);

// device copy of the tables in the layout of LqgTab<n>
int lqg_upload(mpb200_lq *lq) {
    const LqgHost &H = lq->gen;
    size_t bytes = 0;
    void *host = nullptr;
#define PACK(NS_)                                                       \
    case NS_: {                                                         \
        static LqgTab<NS_> tab;                                         \
        lqg_pack<NS_>(H, &tab);                                         \
        host = &tab; bytes = sizeof(tab);                               \
    } break
    switch (H.n) {
        PACK(1); PACK(2); PACK(3); PACK(4); PACK(5); PACK(6);
    default: return fail(MPB200_EARG, "general LQ systems support state dimension 1..6 (got %d)", H.n);
    }
#undef PACK
    if (int rc = lq->gen_dev.reserve(bytes)) return rc;
    cudaStream_t st = ctx().stream;
    MPB_CUDA(cudaMemcpyAsync(lq->gen_dev.p, host, bytes, cudaMemcpyHostToDevice, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    return MPB200_OK;
}

template <int NS>
static int lqg_build(mpb200_samples *s, const mpb200_lq *lq, double r, mpb200_table *tF, mpb200_table *tB) {
    Context &c = ctx();
    cudaStream_t st = c.stream;
    const int64_t N = s->N, nq = s->q1 - s->q0;
    const double *V = s->V.as<double>();
    const LqgTab<NS> *tab = lq->gen_dev.as<LqgTab<NS>>();
    for (mpb200_table *t : {tF, tB}) {
        if (int rc = t->counts.reserve(sizeof(int) * (size_t)(nq + 1))) return rc;
        if (int rc = t->colptr.reserve(sizeof(int64_t) * (size_t)(nq + 1))) return rc;
    }
    const unsigned nb = (unsigned)ceil_div(nq > 0 ? nq : 1, kLqgThreads);
    phase_bank(MPB200_OP_TABLE);
    phase_mark(0);
    if (nq > 0) {
        lqg_inball_kernel<NS, false><<<nb, kLqgThreads, 0, st>>>(V, N, s->q0, nq, tab, r, tF->counts.as<int>(),
                                                                tB->counts.as<int>(), nullptr, nullptr, nullptr, nullptr,
                                                                nullptr, nullptr);
        MPB_LAUNCHED();
    }
    if (int rc = exclusive_scan<int, int64_t>(tF->counts.as<int>(), nq, tF->colptr.as<int64_t>(), (int64_t)1, s->scan_tmp,
                                              c.d_scalar))
        return rc;
    if (int rc = exclusive_scan<int, int64_t>(tB->counts.as<int>(), nq, tB->colptr.as<int64_t>(), (int64_t)1, s->scan_tmp,
                                              c.d_scalar + 1))
        return rc;
    phase_mark(1);
    MPB_CUDA(cudaMemcpyAsync(c.h_scalar, c.d_scalar, sizeof(int64_t) * 2, cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    const int64_t nnzF = c.h_scalar[0], nnzB = c.h_scalar[1];
    if (int rc = tF->rowval.reserve(sizeof(int64_t) * (size_t)(nnzF + 1))) return rc;
    if (int rc = tF->nzval.reserve(sizeof(double) * (size_t)(nnzF + 1))) return rc;
    if (int rc = tB->rowval.reserve(sizeof(int64_t) * (size_t)(nnzB + 1))) return rc;
    if (int rc = tB->nzval.reserve(sizeof(double) * (size_t)(nnzB + 1))) return rc;
    phase_mark(2);
    if (nq > 0 && (nnzF > 0 || nnzB > 0)) {
        lqg_inball_kernel<NS, true><<<nb, kLqgThreads, 0, st>>>(V, N, s->q0, nq, tab, r, nullptr, nullptr,
                                                               tF->colptr.as<int64_t>(), tB->colptr.as<int64_t>(),
                                                               tF->rowval.as<int64_t>(), tF->nzval.as<double>(),
                                                               tB->rowval.as<int64_t>(), tB->nzval.as<double>());
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

#define MPB_LQG_NS(N_, CALL)                                                                         \
    switch (N_) {                                                                                    \
    case 1: CALL(1); break; case 2: CALL(2); break; case 3: CALL(3); break;                          \
    case 4: CALL(4); break; case 5: CALL(5); break; case 6: CALL(6); break;                          \
    default: return fail(MPB200_EARG, "general LQ systems support state dimension 1..6 (got %d)", N_); \
    }

int lqg_inball_build(mpb200_samples *s, const mpb200_lq *lq, double r, mpb200_table *tF, mpb200_table *tB) {
    if (s->d != lq->gen.n) return fail(MPB200_EARG, "sample dimension %d != state dimension %d", s->d, lq->gen.n);
#define CALL(NS_) return lqg_build<NS_>(s, lq, r, tF, tB)
    MPB_LQG_NS(lq->gen.n, CALL);
#undef CALL
    return 0;
}

int lqg_steer_device(const mpb200_lq *lq, const double *dA, const double *dB, int64_t n, double r, double *d_cost,
                     double *d_topt) {
    cudaStream_t st = ctx().stream;
    const unsigned grid = (unsigned)(ceil_div(n, 128) < 148 * 8 ? ceil_div(n, 128) : 148 * 8);
#define CALL(NS_) lqg_steer_kernel<NS_><<<grid, 128, 0, st>>>(dA, dB, n, lq->gen_dev.as<LqgTab<NS_>>(), r, d_cost, d_topt)
    MPB_LQG_NS(lq->gen.n, CALL);
#undef CALL
    MPB_LAUNCHED();
    return 0;
}

int lqg_edges_free_device(const mpb200_samples *s, const mpb200_table *t, const mpb200_lq *lq, double r,
                          const mpb200_obstacles *o, const mpb200_space_desc *ss, uint32_t *d_bits32,
                          unsigned long long *d_checks) {
    SpaceDev S;
    int dw = 0;
    if (int rc = make_space(ss, s->d, &S, &dw)) return rc;
    if (s->d != lq->gen.n) return fail(MPB200_EARG, "sample dimension %d != state dimension %d", s->d, lq->gen.n);
    if (o->kind == 1 && o->d != dw) return fail(MPB200_EARG, "box dimension %d != workspace dimension %d", o->d, dw);
    cudaStream_t st = ctx().stream;
    int64_t blocks = ceil_div(t->ncols > 0 ? t->ncols : 1, 4);
    const unsigned grid = (unsigned)(blocks < (int64_t)ctx().sm_count * 8 ? blocks : (int64_t)ctx().sm_count * 8);
#define CALL(N_, DW_, K_)                                                                                            \
    lqg_edges_free_kernel<N_, DW_, K_><<<grid, 128, 0, st>>>(s->V.as<double>(), t->colptr.as<int64_t>(),             \
                                                             t->rowval.as<int64_t>(), t->ncols, t->col0,             \
                                                             lq->gen_dev.as<LqgTab<N_>>(), r, S, o->table.as<double>(), \
                                                             o->table_words, o->M, d_bits32, d_checks)
    MPB_LQG_DISPATCH(lq->gen.n, dw, o->kind, CALL);
#undef CALL
    MPB_LAUNCHED();
    return 0;
}

int lqg_motions_free_device(const mpb200_lq *lq, double r, const double *dA, const double *dB, int64_t n, int d_state,
                            const mpb200_obstacles *o, const mpb200_space_desc *ss, uint8_t *d_out,
                            unsigned long long *d_checks) {
    SpaceDev S;
    int dw = 0;
    if (int rc = make_space(ss, d_state, &S, &dw)) return rc;
    if (d_state != lq->gen.n) return fail(MPB200_EARG, "state dimension %d != %d", d_state, lq->gen.n);
    if (o->kind == 1 && o->d != dw) return fail(MPB200_EARG, "box dimension %d != workspace dimension %d", o->d, dw);
    cudaStream_t st = ctx().stream;
    const unsigned grid = (unsigned)(ceil_div(n, 128) < 148 * 8 ? ceil_div(n, 128) : 148 * 8);
#define CALL(N_, DW_, K_)                                                                                       \
    lqg_motions_free_kernel<N_, DW_, K_><<<grid, 128, 0, st>>>(dA, dB, n, lq->gen_dev.as<LqgTab<N_>>(), r, S,    \
                                                               o->table.as<double>(), o->M, d_out, d_checks)
    MPB_LQG_DISPATCH(lq->gen.n, dw, o->kind, CALL);
#undef CALL
    MPB_LAUNCHED();
    return 0;
}

}  // namespace mpb
