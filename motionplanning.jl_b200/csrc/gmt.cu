// gmt.cu -- group-marching FMT* (GMT*) over the device-resident neighbour and validity tables
// (mpb200_gmt_plan, mpb200_gmt_plan_lazy, mpb200_gmt_plan_batch; specification in include/mpb200.h and DESIGN.md section 10b).
//
// The planning kernel lives in gmt.cuh.  Table mode instantiates it here with the edge-bit lookup; lazy mode validates
// the arguments it shares with table mode here and hands the launch to the family that owns the motion check
// (gmt_lazy_straight in collide.cu, gmt_lazy_lq in lq.cu, gmt_lazy_lqg in lq_general.cu, gmt_lazy_car in cars.cu).
#include "gmt.cuh"
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <vector>

namespace mpb {

// table mode: step 4 reads the edge bit of the winning entry (the last *_edges_free result on DB)
struct GmtTableEdge {
    static constexpr bool kLazy = false;
    __device__ __forceinline__ bool operator()(const GmtArgs &a, long long e, int, int, GmtCtl *) const {
        return gmt_bit_of(a.ebits, e);
    }
};

int gmt_lazy_straight(const GmtArgs &a, const mpb200_obstacles *o, const mpb200_space_desc *ss, int *blocks);
int gmt_lazy_lq(const GmtArgs &a, const mpb200_lq *lq, double r, const mpb200_obstacles *o, const mpb200_space_desc *ss,
                int *blocks);
int gmt_lazy_lqg(const GmtArgs &a, const mpb200_lq *lq, double r, const mpb200_obstacles *o, const mpb200_space_desc *ss,
                 int *blocks);
int gmt_lazy_car(const GmtArgs &a, int kind, double rturn, double speed, const mpb200_obstacles *o,
                 const mpb200_space_desc *ss, int *blocks);
int car_args(int32_t kind, double rturn, double speed);

int gmt_launch_kernel(const void *kernel, void **args, int *blocks) {
    Context &c = ctx();
    int occ = 0;
    MPB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, kGmtThreads, 0));
    if (occ < 1) return fail(MPB200_ECUDA, "the planning kernel cannot be resident on an SM");
    const int max_blocks = occ * c.sm_count;
    static const int env_grid = [] { const char *e = getenv("MPB200_GMT_GRID"); return e ? atoi(e) : 0; }();
    *blocks = env_grid > 0 ? std::min(env_grid, max_blocks) : std::min(occ, kGmtBlocksPerSM) * c.sm_count;
    phase_bank(MPB200_OP_PLAN);
    phase_mark(0);
    cudaError_t e = cudaLaunchCooperativeKernel(kernel, dim3(*blocks), dim3(kGmtThreads), args, 0, c.stream);
    c.launches++;
    trace_mark(__FILE__, __LINE__);
    phase_mark(1);
    phases_collect(1);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(MPB200_ECUDA, "GMT* planning failed: %s", cudaGetErrorString(e));
    }
    return 0;
}

int gmt_check_roadmap(const mpb200_samples *s, const mpb200_gmt_desc *desc, bool edge_bits) {
    const int64_t N = s->N;
    MPB_CHECK_ARG(s->d <= kMaxDim, "state dimension out of range");
    for (const mpb200_table *t : {desc->fwd, desc->bwd}) {
        MPB_CHECK_ARG(t->src_serial == s->serial && t->src_N == N && t->src_d == s->d,
                      "a table was not built from this sample set");
        MPB_CHECK_ARG(t->col0 == 0 && t->ncols == N, "a table covers a query range other than [0, N) (sharded tables are not supported)");
    }
    const mpb200_table *B = desc->bwd;
    if (edge_bits)
        MPB_CHECK_ARG(B->nnz == 0 || (B->edge_bits_valid && B->edge_bits_nnz == B->nnz),
                      "the backward table has no edge bits for its current contents");
    MPB_CHECK_ARG(!desc->checkpts || s->point_bits_valid, "checkpts needs the point bits of all N samples of this set");
    const mpb200_space_desc *ss = desc->space;
    MPB_CHECK_ARG(!ss || (ss->n == s->d && ss->lo && ss->hi), "space dimension does not match the samples");
    return 0;
}

// edges == NULL: table mode.  A single plan is the batch of one query.
static int gmt_plan(const mpb200_samples *s, const mpb200_gmt_desc *descs, int64_t nq, const mpb200_gmt_edges *edges,
                    mpb200_gmt_result *res, int64_t *segment_checks, int64_t *paths, int64_t path_cap, int64_t *trees,
                    double *costs) {
    MPB_REQUIRE_INIT();
    MPB_CHECK_ARG(s != nullptr && descs != nullptr && res != nullptr, "NULL argument");
    MPB_CHECK_ARG(nq >= 1, "a batch needs at least one query");
    const mpb200_gmt_desc *desc = descs;  // the fields every query shares
    MPB_CHECK_ARG(desc->fwd != nullptr && desc->bwd != nullptr, "fwd and bwd tables are required");
    for (int64_t q = 0; q < nq; ++q) {
        const mpb200_gmt_desc &dq = descs[q];
        MPB_CHECK_ARG(dq.fwd == desc->fwd && dq.bwd == desc->bwd && !dq.checkpts == !desc->checkpts &&
                          dq.space == desc->space,
                      "the queries of a batch must share fwd, bwd, checkpts and space");
        MPB_CHECK_ARG(dq.goal_bits != nullptr, "goal_bits is NULL");
    }
    MPB_CHECK_ARG(path_cap >= 0 && (paths != nullptr || path_cap == 0), "path is NULL with path_cap > 0");
    const int64_t N = s->N;
    MPB_CHECK_ARG(N >= 1, "the sample set is empty");
    for (int64_t q = 0; q < nq; ++q) {
        MPB_CHECK_ARG(descs[q].init >= 1 && descs[q].init <= N, "init out of range (1..N)");
        MPB_CHECK_ARG(descs[q].width >= 0, "width must be a non-negative number");
    }
    if (int rc = gmt_check_roadmap(s, desc, edges == nullptr)) return rc;
    const mpb200_table *B = desc->bwd;
    const mpb200_space_desc *ss = desc->space;
    if (edges) {
        MPB_CHECK_ARG(ss != nullptr, "lazy edge tests need desc->space");
        MPB_CHECK_ARG(edges->obstacles != nullptr, "obstacle handle is NULL");
        if (edges->kind == MPB200_GMT_EDGES_LQ) {
            MPB_CHECK_ARG(edges->lq != nullptr, "LQ edge tests need the LQ system");
            MPB_CHECK_ARG(edges->r > 0 && edges->r < INFINITY, "r must be positive and finite");
        } else if (edges->kind == MPB200_GMT_EDGES_CAR) {
            MPB_CHECK_ARG(s->d == 3, "car spaces need SE2 states (d = 3: x, y, theta)");
            if (int rc = car_args(edges->car_kind, edges->turning_radius, edges->speed)) return rc;
        } else {
            MPB_CHECK_ARG(edges->kind == MPB200_GMT_EDGES_STRAIGHT, "unknown edge kind");
        }
    }

    Context &c = ctx();
    cudaStream_t st = c.stream;
    const int64_t gwords = ceil_div(N, 64);
    const int64_t pcap = std::min(path_cap, N);  // no path is longer than N
    // scratch: C f64 | A i64 | L0, L1, G, X u64 | paths i64 | lists | control blocks | goal masks | status i32, the
    // N-sized arrays nq times (MPB200_GMT_BATCH_BYTES_PER_QUERY in include/mpb200.h)
    static_assert(sizeof(GmtCtl) == 120, "MPB200_GMT_BATCH_BYTES_PER_QUERY counts 120 bytes of control block");
    const size_t per_query = (size_t)N * (8 + 8 + 4 * 8 + 4) + sizeof(int64_t) * pcap + sizeof(GmtCtl) +
                             sizeof(uint64_t) * gwords;
    if (nq > INT_MAX || (size_t)nq > (SIZE_MAX - sizeof(GmtLists)) / per_query)
        return fail(MPB200_ENOMEM, "a batch of %lld queries over %lld samples does not fit in device memory",
                    (long long)nq, (long long)N);
    const size_t nN = (size_t)nq * N;
    const size_t off_A = sizeof(double) * nN, off_L = off_A + sizeof(int64_t) * nN;
    const size_t off_path = off_L + 4 * sizeof(uint64_t) * nN;
    const size_t off_lists = off_path + sizeof(int64_t) * nq * pcap;
    const size_t off_ctl = off_lists + sizeof(GmtLists), off_goal = off_ctl + sizeof(GmtCtl) * nq;
    const size_t off_status = off_goal + sizeof(uint64_t) * gwords * nq;
    DevBuf scratch;
    if (int rc = scratch.reserve(off_status + sizeof(int) * nN)) return rc;
    char *base = scratch.as<char>();

    // lists, control blocks and goal masks start as the host writes them: one copy
    std::vector<char> init(off_status - off_lists);
    GmtLists *hl = reinterpret_cast<GmtLists *>(init.data());
    hl->nopen[0] = (unsigned long long)nq;
    hl->nactive = (int)nq;
    GmtCtl *hc = reinterpret_cast<GmtCtl *>(init.data() + (off_ctl - off_lists));
    for (int64_t q = 0; q < nq; ++q) {
        hc[q].minb[0] = 0;  // C[init] = +0.0
        hc[q].minb[1] = kGmtNone;
        hc[q].goalc = kGmtNone;
        hc[q].goal = INT_MAX;
        hc[q].init = (int)(descs[q].init - 1);
        hc[q].w = descs[q].width;
        memcpy(init.data() + (off_goal - off_lists) + sizeof(uint64_t) * gwords * q, descs[q].goal_bits,
               sizeof(uint64_t) * gwords);
    }

    GmtArgs a = {};
    a.fcp = desc->fwd->colptr.as<int64_t>(); a.frv = desc->fwd->rowval.as<int64_t>();
    a.bcp = B->colptr.as<int64_t>(); a.brv = B->rowval.as<int64_t>(); a.bnz = B->nzval.as<double>();
    a.ebits = edges ? nullptr : B->edge_bits.as<uint32_t>();
    a.pbits = desc->checkpts ? s->point_bits.as<uint32_t>() : nullptr;
    a.gbits = reinterpret_cast<const uint32_t *>(base + off_goal);
    a.gstride = 2 * gwords;
    a.V = s->V.as<double>();
    a.N = (int)N; a.d = s->d; a.nq = (int)nq; a.inb_on = ss != nullptr;
    for (int k = 0; ss && k < s->d; ++k) a.lo[k] = ss->lo[k], a.hi[k] = ss->hi[k];
    a.C = reinterpret_cast<double *>(base); a.A = reinterpret_cast<int64_t *>(base + off_A);
    unsigned long long *L = reinterpret_cast<unsigned long long *>(base + off_L);
    a.L0 = L; a.L1 = L + nN; a.G = L + 2 * nN; a.X = L + 3 * nN;
    a.path = pcap ? reinterpret_cast<int64_t *>(base + off_path) : nullptr;
    a.path_cap = pcap;
    a.lists = reinterpret_cast<GmtLists *>(base + off_lists);
    a.ctl = reinterpret_cast<GmtCtl *>(base + off_ctl);
    a.status = reinterpret_cast<int *>(base + off_status);

    int blocks = 0;
    int rc = 0;
    cudaError_t e = cudaMemcpyAsync(base + off_lists, init.data(), init.size(), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        if (!edges) rc = gmt_launch(a, GmtTableEdge{}, &blocks);
        else if (edges->kind == MPB200_GMT_EDGES_STRAIGHT) rc = gmt_lazy_straight(a, edges->obstacles, ss, &blocks);
        else if (edges->kind == MPB200_GMT_EDGES_LQ)
            rc = (edges->lq->general ? gmt_lazy_lqg : gmt_lazy_lq)(a, edges->lq, edges->r, edges->obstacles, ss, &blocks);
        else rc = gmt_lazy_car(a, edges->car_kind, edges->turning_radius, edges->speed, edges->obstacles, ss, &blocks);
    }
    if (rc) {
        scratch.release();
        return rc;
    }
    std::vector<GmtCtl> h(nq);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h.data(), a.ctl, sizeof(GmtCtl) * nq, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && trees) e = cudaMemcpyAsync(trees, a.A, sizeof(int64_t) * nN, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && costs) e = cudaMemcpyAsync(costs, a.C, sizeof(double) * nN, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    bool copied = false;
    for (int64_t q = 0; q < nq && e == cudaSuccess; ++q) {
        if (h[q].path_len > 0 && h[q].path_len <= pcap) {
            e = cudaMemcpyAsync(paths + q * path_cap, a.path + q * pcap, sizeof(int64_t) * h[q].path_len,
                                cudaMemcpyDeviceToHost, st);
            copied = true;
        }
    }
    if (e == cudaSuccess && copied) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
        cudaGetLastError();
        rc = fail(MPB200_ECUDA, "GMT* planning failed: %s", cudaGetErrorString(e));
    }
    scratch.release();
    if (rc) return rc;
    for (int64_t q = 0; q < nq; ++q) {
        res[q].solved = h[q].solved;
        res[q].grid_blocks = blocks;
        res[q].goal = h[q].goal1;
        res[q].cost = h[q].cost;
        res[q].iterations = h[q].iterations;
        res[q].expansions = h[q].expansions;
        res[q].checks = (int64_t)h[q].checks;
        res[q].checks_in_bounds = (int64_t)h[q].checks_inb;
        res[q].path_len = h[q].path_len;
        if (segment_checks) segment_checks[q] = (int64_t)h[q].segs;
    }
    return MPB200_OK;
}

}  // namespace mpb

using namespace mpb;

extern "C" {

int mpb200_gmt_plan(const mpb200_samples *s, const mpb200_gmt_desc *desc, mpb200_gmt_result *res, int64_t *path,
                    int64_t path_cap, int64_t *tree, double *costs) {
    return gmt_plan(s, desc, 1, nullptr, res, nullptr, path, path_cap, tree, costs);
}

int mpb200_gmt_plan_lazy(const mpb200_samples *s, const mpb200_gmt_desc *desc, const mpb200_gmt_edges *edges,
                         mpb200_gmt_result *res, int64_t *segment_checks, int64_t *path, int64_t path_cap,
                         int64_t *tree, double *costs) {
    MPB_CHECK_ARG(edges != nullptr, "edges is NULL");
    return gmt_plan(s, desc, 1, edges, res, segment_checks, path, path_cap, tree, costs);
}

int mpb200_gmt_plan_batch(const mpb200_samples *s, const mpb200_gmt_desc *descs, int64_t nq,
                          const mpb200_gmt_edges *edges, mpb200_gmt_result *res, int64_t *segment_checks,
                          int64_t *paths, int64_t path_cap, int64_t *trees, double *costs) {
    return gmt_plan(s, descs, nq, edges, res, segment_checks, paths, path_cap, trees, costs);
}

}  // extern "C"
