// lq_general.cuh -- device side of the general linear-affine LQ path (lq_general.cu): the per-system tables, the
// 2BVP evaluated operation for operation as oracle/lq_general.c specifies, the K9 motion check and the compiled
// (state dim, workspace dim, checker kind) combinations.  Shared by lq_general.cu and the lazy GMT* planner
// (gmt_lqg.cu).
#pragma once
#include "common.cuh"
#include "predicates.cuh"
#include <cmath>

namespace mpb {

template <int NS>
struct LqgTab {
    double A[NS * NS], c[NS], BRB[NS * NS];
    double Ak[NS][NS * NS], dk[NS][NS];
    double Gp[2 * NS - 1][NS * NS];
};

// ---- device: the oracle's evaluation, operation for operation ---------------------------------------------
template <int NS>
__device__ __forceinline__ void lqg_xbar(const LqgTab<NS> &S, const double *x, double t, double *xb) {
    double tp = 1.0;
#pragma unroll
    for (int i = 0; i < NS; ++i) xb[i] = 0.0;
#pragma unroll
    for (int k = 0; k < NS; ++k) {
        const double tp1 = dmul(tp, t);
#pragma unroll
        for (int i = 0; i < NS; ++i) {
            double s = 0.0;
#pragma unroll
            for (int j = 0; j < NS; ++j) s = dadd(s, dmul(S.Ak[k][i * NS + j], x[j]));
            xb[i] = dadd(xb[i], dadd(dmul(s, tp), dmul(S.dk[k][i], tp1)));
        }
        tp = tp1;
    }
}
template <int NS>
__device__ __forceinline__ void lqg_G(const LqgTab<NS> &S, double t, double *G) {
#pragma unroll
    for (int i = 0; i < NS * NS; ++i) G[i] = 0.0;
    double tp = 1.0;
#pragma unroll
    for (int p = 0; p < 2 * NS - 1; ++p) {
        tp = dmul(tp, t);
#pragma unroll
        for (int i = 0; i < NS * NS; ++i) G[i] = dadd(G[i], dmul(S.Gp[p][i], tp));
    }
}
template <int NS>
__device__ __forceinline__ bool lqg_chol(const double *G, double *Lw) {
    bool ok = true;
#pragma unroll
    for (int i = 0; i < NS; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            double s = G[i * NS + j];
#pragma unroll
            for (int k = 0; k < j; ++k) s = dsub(s, dmul(Lw[i * NS + k], Lw[j * NS + k]));
            if (i == j) {
                if (!(s > 0)) ok = false;
                Lw[i * NS + i] = __dsqrt_rn(s);
            } else {
                Lw[i * NS + j] = ddiv(s, Lw[j * NS + j]);
            }
        }
    return ok;
}
template <int NS>
__device__ __forceinline__ void lqg_chol_solve(const double *Lw, const double *b, double *x) {
    double y[NS];
#pragma unroll
    for (int i = 0; i < NS; ++i) {
        double s = b[i];
#pragma unroll
        for (int k = 0; k < i; ++k) s = dsub(s, dmul(Lw[i * NS + k], y[k]));
        y[i] = ddiv(s, Lw[i * NS + i]);
    }
#pragma unroll
    for (int i = NS - 1; i >= 0; --i) {
        double s = y[i];
#pragma unroll
        for (int k = i + 1; k < NS; ++k) s = dsub(s, dmul(Lw[k * NS + i], x[k]));
        x[i] = ddiv(s, Lw[i * NS + i]);
    }
}
// (cost, dcost, ddcost); G(t) not numerically positive definite -> (+inf, 1, 0) like the oracle
template <int NS>
__device__ __noinline__ void lqg_terms(const LqgTab<NS> &S, const double *x, const double *y, double t, double *out3) {
    double xb[NS], e[NS], G[NS * NS], Lw[NS * NS], lam[NS], f[NS], h[NS], mu[NS], bl[NS];
    lqg_xbar<NS>(S, x, t, xb);
#pragma unroll
    for (int i = 0; i < NS; ++i) e[i] = dsub(y[i], xb[i]);
    lqg_G<NS>(S, t, G);
    if (!lqg_chol<NS>(G, Lw)) {
        out3[0] = __longlong_as_double(0x7ff0000000000000LL); out3[1] = 1.0; out3[2] = 0.0;
        return;
    }
    lqg_chol_solve<NS>(Lw, e, lam);
#pragma unroll
    for (int i = 0; i < NS; ++i) {
        double s = 0.0, b = 0.0;
#pragma unroll
        for (int j = 0; j < NS; ++j) {
            s = dadd(s, dmul(S.A[i * NS + j], y[j]));
            b = dadd(b, dmul(S.BRB[i * NS + j], lam[j]));
        }
        f[i] = dadd(s, S.c[i]);
        bl[i] = b;
        h[i] = dadd(f[i], b);
    }
    lqg_chol_solve<NS>(Lw, h, mu);
    double el = 0.0, lf = 0.0, lb = 0.0, dd = 0.0;
#pragma unroll
    for (int i = 0; i < NS; ++i) {
        double atl = 0.0;
#pragma unroll
        for (int j = 0; j < NS; ++j) atl = dadd(atl, dmul(S.A[j * NS + i], lam[j]));
        el = dadd(el, dmul(e[i], lam[i]));
        lf = dadd(lf, dmul(lam[i], f[i]));
        lb = dadd(lb, dmul(lam[i], bl[i]));
        dd = dadd(dd, dmul(dadd(mu[i], atl), h[i]));
    }
    out3[0] = dadd(t, el);
    out3[1] = dsub(dsub(1.0, dmul(2.0, lf)), lb);
    out3[2] = dmul(2.0, dd);
}
template <int NS>
__device__ __forceinline__ double lqg_dcost(const LqgTab<NS> &S, const double *x, const double *y, double t) {
    double o[3];
    lqg_terms<NS>(S, x, y, t, o);
    return o[1];
}
template <int NS>
__device__ __forceinline__ double lqg_topt_newton(const LqgTab<NS> &S, const double *x, const double *y, double tm) {
    const double tol = 1e-6;
    double b = tm;
    if (lqg_dcost<NS>(S, x, y, b) < 0) return tm;
    double a = ddiv(tm, 100.0);
    for (int k = 0; k < 60 && lqg_dcost<NS>(S, x, y, a) > 0; ++k) a = ddiv(a, 2.0);
    double t = ddiv(tm, 2.0);
    double o[3];
    lqg_terms<NS>(S, x, y, t, o);
    double cdval = o[1];
    int it = 0;
    while (fabs(cdval) > tol && fabs(dsub(a, b)) > tol) {
        t = dsub(t, ddiv(cdval, o[2]));
        if (!(t >= a && t <= b)) t = ddiv(dadd(a, b), 2.0);
        lqg_terms<NS>(S, x, y, t, o);
        cdval = o[1];
        if (cdval > 0) b = t; else a = t;
        if (++it >= 200) break;
    }
    return t;
}
template <int NS>
__device__ __forceinline__ bool lqg_same(const double *x0, const double *x1) {
    bool same = true;
#pragma unroll
    for (int i = 0; i < NS; ++i) same = same && (x0[i] == x1[i]);
    return same;
}
template <int NS>
__device__ __forceinline__ void lqg_steer(const LqgTab<NS> &S, const double *x0, const double *x1, double r, double *cost,
                                          double *topt) {
    if (lqg_same<NS>(x0, x1)) { *cost = 0.0; *topt = 0.0; return; }
    const double t = lqg_topt_newton<NS>(S, x0, x1, r);
    double o[3];
    lqg_terms<NS>(S, x0, x1, t, o);
    *cost = o[0];
    *topt = t;
}
template <int NS>
__device__ __noinline__ void lqg_state(const LqgTab<NS> &S, const double *x0, const double *x1, double t, double s,
                                       double *out) {
    double xb[NS], e[NS], G[NS * NS], Lw[NS * NS], lam[NS], w[NS];
    lqg_xbar<NS>(S, x0, t, xb);
#pragma unroll
    for (int i = 0; i < NS; ++i) e[i] = dsub(x1[i], xb[i]);
    lqg_G<NS>(S, t, G);
    if (!lqg_chol<NS>(G, Lw)) {
#pragma unroll
        for (int i = 0; i < NS; ++i) out[i] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    lqg_chol_solve<NS>(Lw, e, lam);
    const double ts = dsub(t, s);
    double tp = 1.0;
#pragma unroll
    for (int i = 0; i < NS; ++i) w[i] = 0.0;
#pragma unroll
    for (int k = 0; k < NS; ++k) {
#pragma unroll
        for (int i = 0; i < NS; ++i) {
            double a = 0.0;
#pragma unroll
            for (int j = 0; j < NS; ++j) a = dadd(a, dmul(S.Ak[k][j * NS + i], lam[j]));
            w[i] = dadd(w[i], dmul(a, tp));
        }
        tp = dmul(tp, ts);
    }
    lqg_xbar<NS>(S, x0, s, xb);
    lqg_G<NS>(S, s, G);
#pragma unroll
    for (int i = 0; i < NS; ++i) {
        double a = 0.0;
#pragma unroll
        for (int j = 0; j < NS; ++j) a = dadd(a, dmul(G[i * NS + j], w[j]));
        out[i] = dadd(xb[i], a);
    }
}

template <int NS>
__device__ __forceinline__ const LqgTab<NS> &lqg_stage(const LqgTab<NS> *g, LqgTab<NS> *s) {
    const double *src = reinterpret_cast<const double *>(g);
    double *dst = reinterpret_cast<double *>(s);
    for (int i = threadIdx.x; i < (int)(sizeof(LqgTab<NS>) / sizeof(double)); i += blockDim.x) dst[i] = src[i];
    __syncthreads();
    return *s;
}

constexpr int kLqgThreads = 128;
constexpr int kLqgTile = 64;

// K5, general form.  FILL = false: per-column counts for both directions; true: rows + costs.
// K9, general form: is_free_motion(v, w, CC, SS) along the optimal trajectory (5 waypoints)
template <int NS, int DW, int KIND>
__device__ __forceinline__ bool lqg_motion_free(const LqgTab<NS> &L, const SpaceDev &S, const double *T, int M, double r,
                                                const double *v, const double *w, int *checks) {
    double c, t;
    lqg_steer<NS>(L, v, w, r, &c, &t);
    double cur[NS], nxt[NS], p[DW], q[DW];
    if (t == 0.0) {
#pragma unroll
        for (int k = 0; k < NS; ++k) cur[k] = v[k];
    } else {
        lqg_state<NS>(L, v, w, t, 0.0, cur);
    }
    state2workspace<NS, DW>(S, cur, p);
    for (int i = 1; i <= 4; ++i) {
        if (!in_state_space<NS>(S, cur)) return false;  // only wps[1..4] are bounds-checked (Q4)
        const double s = ddiv(dmul((double)i, t), 4.0);
        if (t == 0.0) {
#pragma unroll
            for (int k = 0; k < NS; ++k) nxt[k] = v[k];
        } else {
            lqg_state<NS>(L, v, w, t, s, nxt);
        }
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

// (state dim, workspace dim, checker kind) combinations compiled for the general path
#define MPB_LQG_DISPATCH(N_, DW_, KIND_, CALL)                                                            \
    do {                                                                                                  \
        if (KIND_ == 0 && DW_ != 2) return fail(MPB200_EARG, "2-D obstacles need a 2-D workspace");       \
        if (N_ == 4 && DW_ == 2 && KIND_ == 0) { CALL(4, 2, 0); }                                         \
        else if (N_ == 4 && DW_ == 2 && KIND_ == 1) { CALL(4, 2, 1); }                                    \
        else if (N_ == 6 && DW_ == 3 && KIND_ == 1) { CALL(6, 3, 1); }                                    \
        else if (N_ == 6 && DW_ == 2 && KIND_ == 0) { CALL(6, 2, 0); }                                    \
        else if (N_ == 2 && DW_ == 1 && KIND_ == 1) { CALL(2, 1, 1); }                                    \
        else if (N_ == 3 && DW_ == 1 && KIND_ == 1) { CALL(3, 1, 1); }                                    \
        else if (N_ == 3 && DW_ == 2 && KIND_ == 0) { CALL(3, 2, 0); }                                    \
        else if (N_ == 2 && DW_ == 2 && KIND_ == 0) { CALL(2, 2, 0); }                                    \
        else return fail(MPB200_EARG, "unsupported general-LQ (n=%d, workspace=%d, checker=%d) combination", N_, DW_, KIND_); \
    } while (0)

}  // namespace mpb
