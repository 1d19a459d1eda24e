// gmt_lqg.cu -- lazy GMT* over general linear-affine LQ systems: the planning kernel of gmt.cuh with the K9 motion check
// of lq_general.cuh as its edge test.  A translation unit of its own: instantiated inside lq_general.cu these kernels
// would change the register convention of the non-inlined helpers that module's existing kernels share.
#include "lq_general.cuh"
#include "gmt.cuh"

namespace mpb {

int make_space(const mpb200_space_desc *ss, int d_state, SpaceDev *out, int *dw);

// lazy GMT*: step 4 runs lqg_motion_free (the check of lqg_edges_free_kernel) on the winning entry, on one lane; the
// system tables and the obstacle table are read through L1
template <int NS, int DW, int KIND>
struct GmtLqgEdge {
    static constexpr bool kLazy = true;
    const LqgTab<NS> *L;
    double r;
    SpaceDev S;
    const double *T;
    int M;
    __device__ bool operator()(const GmtArgs &a, long long, int y, int x, GmtCtl *ctl) const {
        double v[NS], w[NS];
        gmt_endpoints<NS>(a, y, x, v, w);
        int nchk = 0;
        const bool ok = lqg_motion_free<NS, DW, KIND>(*L, S, T, M, r, v, w, &nchk);
        gmt_count_segments(ctl, nchk);
        return ok;
    }
};

int gmt_lazy_lqg(const GmtArgs &a, const mpb200_lq *lq, double r, const mpb200_obstacles *o, const mpb200_space_desc *ss,
                 int *blocks) {
    SpaceDev S;
    int dw = 0;
    if (int rc = make_space(ss, a.d, &S, &dw)) return rc;
    if (a.d != lq->gen.n) return fail(MPB200_EARG, "sample dimension %d != state dimension %d", a.d, lq->gen.n);
    if (o->kind == 1 && o->d != dw) return fail(MPB200_EARG, "box dimension %d != workspace dimension %d", o->d, dw);
#define CALL(N_, DW_, K_)                                                                                                  \
    return gmt_launch(a, GmtLqgEdge<N_, DW_, K_>{lq->gen_dev.as<LqgTab<N_>>(), r, S, o->table.as<double>(), o->M}, blocks)
    MPB_LQG_DISPATCH(lq->gen.n, dw, o->kind, CALL);
#undef CALL
    return 0;
}

}  // namespace mpb
