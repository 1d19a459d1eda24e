// cars.cu -- chopped-metric car spaces: Dubins / Reeds-Shepp exact steering as batched device code.
//
// Replaces, for every stored pair at once, the reference's per-call
//   dubins / reedsshepp                         src/statespaces/simplecars.jl:102-213, 230-523
//   evaluate(::ChoppedPreMetric, v, w)          src/primitivetypes.jl:95-100
//   inball(V, ::ChoppedPreMetric, ::TreeDistanceDS, v, r, forwards)   src/nearneighbors.jl:185-198
//     (KD-tree over (x, y) as the lower bound, simplecars.jl:42-52 -> here: the grid r-ball table K1 + K2 over
//      the (x, y) columns supplies the candidates, this file evaluates the exact metric on them and compacts)
//   propagate / collision_waypoints             simplecars.jl:55-82, statespaces.jl:134-142
//   is_free_motion(v, w, CC, SS)                statespaces.jl:153-158
//
// Arithmetic: IEEE double in the reference's operation order; this translation unit is compiled with -fmad=false
// (build.py), so no multiply-add is contracted.  sin / cos / atan2 / acos are the fixed routines specified in
// oracle/cars.c (the reference's openlibm calls are not reproducible: parity unpinned there), sqrt and division are
// correctly rounded, mod2piF is exact (an explicit fma recovers the remainder).
#include "common.cuh"
#include "predicates.cuh"
#include "scan.cuh"
#include "gmt.cuh"
#include <algorithm>
#include <limits>

namespace mpb {

namespace car {

constexpr double kPi = 3.141592653589793;
constexpr double kTwoPi = 6.283185307179586;
constexpr double kInf = __builtin_huge_val();

// Julia's mod(x, 2pi): exact remainder with the sign of the divisor.  The quotient comes from a multiplication by
// 1/2pi (it can be off by one next to an integer); x - q*2pi is then exact in one fma (a multiple of ulp(2pi) below 8
// whenever q is within one of the true quotient), and a wrong q is corrected and the remainder recomputed, so the
// result equals fmod(x, 2pi) bit for bit (the oracle calls libm's fmod).
__device__ __forceinline__ double mod2pi(double x) {
    double q = trunc(x * 0.15915494309189535);
    double r = __fma_rn(-q, kTwoPi, x);
    const bool pos = x >= 0.0;
    const bool down = pos ? (r < 0.0) : (r <= -kTwoPi);   // quotient one too large in magnitude towards +inf
    const bool up = pos ? (r >= kTwoPi) : (r > 0.0);
    if (down || up) {                                      // rare: x / 2pi rounded across an integer
        q += up ? 1.0 : -1.0;
        r = __fma_rn(-q, kTwoPi, x);
    }
    if (r == 0.0) return 0.0;
    return r < 0.0 ? r + kTwoPi : r;
}

__device__ __noinline__ void sincos_(double x, double *sn, double *cs) {
    // on |x|, reflected: sin is exactly odd and cos exactly even (evaluations at -t are shared with those at t)
    const double ax = fabs(x);
    const double kf = floor(ax * 0.6366197723675814 + 0.5);
    const double th = ((ax - kf * 1.5707963267341256) - kf * 6.077100506303966e-11) - kf * 2.0222662487111665e-21;
    const double t2 = th * th;
    double ps = -1.0 / 355687428096000.0;
    ps = ps * t2 + 1.0 / 1307674368000.0;
    ps = ps * t2 - 1.0 / 6227020800.0;
    ps = ps * t2 + 1.0 / 39916800.0;
    ps = ps * t2 - 1.0 / 362880.0;
    ps = ps * t2 + 1.0 / 5040.0;
    ps = ps * t2 - 1.0 / 120.0;
    ps = ps * t2 + 1.0 / 6.0;
    const double s = th - th * t2 * ps;
    double pc = 1.0 / 6402373705728000.0;
    pc = pc * t2 - 1.0 / 20922789888000.0;
    pc = pc * t2 + 1.0 / 87178291200.0;
    pc = pc * t2 - 1.0 / 479001600.0;
    pc = pc * t2 + 1.0 / 3628800.0;
    pc = pc * t2 - 1.0 / 40320.0;
    pc = pc * t2 + 1.0 / 720.0;
    pc = pc * t2 - 1.0 / 24.0;
    pc = pc * t2 + 0.5;
    const double c = 1.0 - t2 * pc;
    const int q = (int)((long long)kf & 3);
    // quadrant by selects (no divergence): q = 0: (s, c)  1: (c, -s)  2: (-s, -c)  3: (-c, s)
    const double a = (q & 1) ? c : s, b = (q & 1) ? s : c;
    const double sq = (q & 2) ? -a : a;
    *cs = ((q + 1) & 2) ? -b : b;
    *sn = (x < 0.0) ? -sq : sq;
}

__device__ __forceinline__ double atan01(double a) {
    const int ci = (int)(a * 4.0 + 0.5);
    const double c = 0.25 * (double)ci;
    const double t = (a - c) / (1.0 + a * c);
    const double t2 = t * t;
    double p = 1.0 / 21.0;
    p = 1.0 / 19.0 - p * t2;
    p = 1.0 / 17.0 - p * t2;
    p = 1.0 / 15.0 - p * t2;
    p = 1.0 / 13.0 - p * t2;
    p = 1.0 / 11.0 - p * t2;
    p = 1.0 / 9.0 - p * t2;
    p = 1.0 / 7.0 - p * t2;
    p = 1.0 / 5.0 - p * t2;
    p = 1.0 / 3.0 - p * t2;
    p = 1.0 - p * t2;
    const double base = ci == 0 ? 0.0 : ci == 1 ? 0.24497866312686414 : ci == 2 ? 0.4636476090008061
                      : ci == 3 ? 0.6435011087932844 : 0.7853981633974483;
    return base + t * p;
}
__device__ __noinline__ double atan2_(double y, double x) {
    const double ax = fabs(x), ay = fabs(y);
    // one evaluation of the [0, 1] kernel on min / max, then selects (the same values as the two-branch form)
    const bool swap = !(ay <= ax);
    const double num = swap ? ax : ay, den = swap ? ay : ax;
    const bool zero = ax == 0.0 && ay == 0.0;
    double ang = atan01(zero ? 0.0 : num / den);
    if (swap) ang = 1.5707963267948966 - ang;
    if (zero) ang = 0.0;
    if (signbit(x)) ang = kPi - ang;
    return signbit(y) ? -ang : ang;
}
__device__ __forceinline__ double acos_(double x) {
    double rad = (1.0 - x) * (1.0 + x);
    if (rad < 0.0) rad = 0.0;
    return atan2_(sqrt(rad), x);
}

struct Seg { double t, u1, u2; };
__device__ __forceinline__ Seg mkseg(int turn, double d) {
    Seg s;
    s.t = fabs(d);
    s.u1 = d > 0.0 ? 1.0 : (d < 0.0 ? -1.0 : 0.0);
    s.u2 = (double)turn;
    return s;
}
struct Best { double c; int l; Seg p[5]; };

// ---- Dubins (simplecars.jl:102-194): the six words in the reference's order ------------------------------------
// word: 0 LSL 1 RSR 2 RSL 3 LSR 4 RLR 5 LRL
__device__ __forceinline__ void dubins_word(int word, double d, double a, double b, double ca, double sa, double cb,
                                            double sb, Best &B) {
    double t, p, q;
    int t0, t1, t2;
    if (word == 0) {
        const double tmp = 2.0 + d * d - 2.0 * (ca * cb + sa * sb - d * (sa - sb));
        if (tmp < 0.0) return;
        const double th = atan2_(cb - ca, d + sa - sb);
        t = mod2pi(-a + th); p = sqrt(tmp > 0.0 ? tmp : 0.0); q = mod2pi(b - th);
        t0 = 1; t1 = 0; t2 = 1;
    } else if (word == 1) {
        const double tmp = 2.0 + d * d - 2.0 * (ca * cb + sa * sb - d * (sb - sa));
        if (tmp < 0.0) return;
        const double th = atan2_(ca - cb, d - sa + sb);
        t = mod2pi(a - th); p = sqrt(tmp > 0.0 ? tmp : 0.0); q = mod2pi(-b + th);
        t0 = -1; t1 = 0; t2 = -1;
    } else if (word == 2) {
        const double tmp = d * d - 2.0 + 2.0 * (ca * cb + sa * sb - d * (sa + sb));
        if (tmp < 0.0) return;
        p = sqrt(tmp > 0.0 ? tmp : 0.0);
        const double th = atan2_(ca + cb, d - sa - sb) - atan2_(2.0, p);
        t = mod2pi(a - th); q = mod2pi(b - th);
        t0 = -1; t1 = 0; t2 = 1;
    } else if (word == 3) {
        const double tmp = -2.0 + d * d + 2.0 * (ca * cb + sa * sb + d * (sa + sb));
        if (tmp < 0.0) return;
        p = sqrt(tmp > 0.0 ? tmp : 0.0);
        const double th = atan2_(-ca - cb, d + sa + sb) - atan2_(-2.0, p);
        t = mod2pi(-a + th); q = mod2pi(-b + th);
        t0 = 1; t1 = 0; t2 = -1;
    } else if (word == 4) {
        const double tmp = (6.0 - d * d + 2.0 * (ca * cb + sa * sb + d * (sa - sb))) / 8.0;
        if (fabs(tmp) >= 1.0) return;
        p = kTwoPi - acos_(tmp);
        const double th = atan2_(ca - cb, d - sa + sb);
        t = mod2pi(a - th + p / 2.0); q = mod2pi(a - b - t + p);
        t0 = -1; t1 = 1; t2 = -1;
    } else {
        const double tmp = (6.0 - d * d + 2.0 * (ca * cb + sa * sb - d * (sa - sb))) / 8.0;
        if (fabs(tmp) >= 1.0) return;
        p = kTwoPi - acos_(tmp);
        const double th = atan2_(-ca + cb, d + sa - sb);
        t = mod2pi(-a + th + p / 2.0); q = mod2pi(b - a - t + p);
        t0 = 1; t1 = -1; t2 = 1;
    }
    const double cnew = t + p + q;
    if (B.c <= cnew) return;
    B.p[0] = mkseg(t0, t); B.p[1] = mkseg(t1, p); B.p[2] = mkseg(t2, q);
    B.c = cnew; B.l = 3;
}

__device__ __forceinline__ void scale_segments(Best &B, double r, double s) {
    for (int i = 0; i < B.l; ++i) {
        B.p[i].t = B.p[i].t * r; B.p[i].u2 = B.p[i].u2 / r;
        B.p[i].t = B.p[i].t / s; B.p[i].u1 = B.p[i].u1 * s;
    }
}

__device__ double dubins(const double *s1, const double *s2, double r, double s, Best &B) {
    const double vx = (s2[0] - s1[0]) / r, vy = (s2[1] - s1[1]) / r;
    const double d = sqrt(vx * vx + vy * vy);
    const double th = atan2_(vy, vx);
    const double a = mod2pi(s1[2] - th), b = mod2pi(s2[2] - th);
    double ca, sa, cb, sb;
    sincos_(a, &sa, &ca);
    sincos_(b, &sb, &cb);
    B.c = kInf; B.l = 3;
    for (int i = 0; i < 5; ++i) B.p[i] = mkseg(0, 0.0);
    for (int word = 0; word < 6; ++word) dubins_word(word, d, a, b, ca, sa, cb, sb, B);
    scale_segments(B, r, s);
    return B.c * r;
}

// ---- Reeds-Shepp (simplecars.jl:215-523) -------------------------------------------------------------------------
__device__ __forceinline__ void Rpolar(double x, double y, double *r, double *th) { *r = sqrt(x * x + y * y); *th = atan2_(y, x); }
__device__ __forceinline__ double Mwrap(double t) { const double m = mod2pi(t); return m > kPi ? m - kTwoPi : m; }
// Tau(u, v, E, N) for v = +-u, given (su, cu) = sincos(u): cos(v) == cos(u) exactly, sin / cos of delta in one call
__device__ double Tau(double u, double v, double E, double N, double su, double cu) {
    const double delta = Mwrap(u - v);
    double sd, cd;
    sincos_(delta, &sd, &cd);
    const double A = su - sd;
    const double Bc = cu - cd - 1.0;
    const double th = atan2_(N * A - E * Bc, E * A + N * Bc);
    const double t = 2.0 * cd - 2.0 * cu - 2.0 * cu + 3.0;
    return t < 0.0 ? Mwrap(th + kPi) : Mwrap(th);
}

// family: 0 LpSpLp 1 LpSpRp 2 LpRmLp 3 LpRmLm 4 LpRpuLmuRm 5 LpRmuLmuRp 6 LpRmSmLm 7 LpRmSmRm 8 LpRmSmLmRp
__device__ bool rs_family(int fam, double tx, double ty, double tt, double stt, double ctt, Best &B) {
    double cnew;
    Seg p0, p1, p2, p3 = mkseg(0, 0.0), p4 = mkseg(0, 0.0);
    int l;
    if (fam == 0) {
        double r, th;
        Rpolar(tx - stt, ty - 1.0 + ctt, &r, &th);
        const double u = r, t = mod2pi(th), v = mod2pi(tt - t);
        cnew = t + u + v;
        p0 = mkseg(1, t); p1 = mkseg(0, u); p2 = mkseg(1, v); l = 3;
    } else if (fam == 1) {
        double r, th, r1, th1;
        Rpolar(tx + stt, ty - 1.0 - ctt, &r, &th);
        if (r * r < 4.0) return false;
        const double u = sqrt(r * r - 4.0);
        Rpolar(u, 2.0, &r1, &th1);
        const double t = mod2pi(th + th1), v = mod2pi(t - tt);
        cnew = t + u + v;
        p0 = mkseg(1, t); p1 = mkseg(0, u); p2 = mkseg(-1, v); l = 3;
    } else if (fam == 2 || fam == 3) {
        const double E = tx - stt, N = ty + ctt - 1.0;
        if (E * E + N * N > 16.0) return false;
        double r, th;
        Rpolar(E, N, &r, &th);
        double u = acos_(1.0 - r * r / 8.0);
        const double t = mod2pi(th - u / 2.0 + kPi);
        double v = mod2pi(kPi - u / 2.0 - th + tt);
        if (fam == 3) v = v - kTwoPi;
        u = -u;
        cnew = fam == 2 ? t - u + v : t - u - v;
        p0 = mkseg(1, t); p1 = mkseg(-1, u); p2 = mkseg(1, v); l = 3;
    } else if (fam == 4) {
        const double E = tx + stt, N = ty - ctt - 1.0;
        const double p = (2.0 + sqrt(E * E + N * N)) / 4.0;
        if (p < 0.0 || p > 1.0) return false;
        const double u = acos_(p);
        double su, cu;
        sincos_(u, &su, &cu);
        const double tau = Tau(u, -u, E, N, su, cu);   // Omega(u, v, E, N, t) = M(Tau(u, v, E, N) - u + v - t)
        const double t = mod2pi(tau);
        const double v = mod2pi(Mwrap(tau - u + (-u) - tt)) - kTwoPi;
        cnew = t + 2.0 * u - v;
        p0 = mkseg(1, t); p1 = mkseg(-1, u); p2 = mkseg(1, -u); p3 = mkseg(-1, v); l = 4;
    } else if (fam == 5) {
        const double E = tx + stt, N = ty - ctt - 1.0;
        const double p = (20.0 - E * E - N * N) / 16.0;
        if (p < 0.0 || p > 1.0) return false;
        const double u = -acos_(p);
        double su, cu;
        sincos_(u, &su, &cu);
        const double tau = Tau(u, u, E, N, su, cu);
        const double t = mod2pi(tau);
        const double v = mod2pi(Mwrap(tau - u + u - tt));
        cnew = t - 2.0 * u + v;
        p0 = mkseg(1, t); p1 = mkseg(-1, u); p2 = mkseg(1, u); p3 = mkseg(-1, v); l = 4;
    } else if (fam == 6) {
        const double E = tx - stt, N = ty + ctt - 1.0;
        double D, beta;
        Rpolar(E, N, &D, &beta);
        if (D < 2.0) return false;
        const double gamma = acos_(2.0 / D);
        const double F = sqrt(D * D / 4.0 - 1.0);
        const double t = mod2pi(kPi + beta - gamma);
        const double u = 2.0 - 2.0 * F;
        if (u > 0.0) return false;
        const double v = mod2pi(-3.0 * kPi / 2.0 + gamma + tt - beta) - kTwoPi;
        cnew = t + kPi / 2.0 - u - v;
        p0 = mkseg(1, t); p1 = mkseg(-1, -kPi / 2.0); p2 = mkseg(0, u); p3 = mkseg(1, v); l = 4;
    } else if (fam == 7) {
        const double E = tx + stt, N = ty - ctt - 1.0;
        double D, beta;
        Rpolar(E, N, &D, &beta);
        if (D < 2.0) return false;
        const double t = mod2pi(beta + kPi / 2.0);
        const double u = 2.0 - D;
        if (u > 0.0) return false;
        const double v = mod2pi(-kPi - tt + beta) - kTwoPi;
        cnew = t + kPi / 2.0 - u - v;
        p0 = mkseg(1, t); p1 = mkseg(-1, -kPi / 2.0); p2 = mkseg(0, u); p3 = mkseg(-1, v); l = 4;
    } else {
        const double E = tx + stt, N = ty - ctt - 1.0;
        double D, beta;
        Rpolar(E, N, &D, &beta);
        if (D < 2.0) return false;
        const double gamma = acos_(2.0 / D);
        const double F = sqrt(D * D / 4.0 - 1.0);
        const double t = mod2pi(kPi + beta - gamma);
        const double u = 4.0 - 2.0 * F;
        if (u > 0.0) return false;
        const double v = mod2pi(kPi + beta - tt - gamma);
        cnew = t + kPi - u + v;
        p0 = mkseg(1, t); p1 = mkseg(-1, -kPi / 2.0); p2 = mkseg(0, u); p3 = mkseg(1, -kPi / 2.0); p4 = mkseg(-1, v); l = 5;
    }
    if (B.c <= cnew) return false;
    B.p[0] = p0; B.p[1] = p1; B.p[2] = p2;
    if (l > 3) B.p[3] = p3;
    if (l > 4) B.p[4] = p4;
    B.c = cnew; B.l = l;
    return true;
}

// the sweep of simplecars.jl:283-339: per family the transformed targets tried, as a bit mask over
// (0 target, 1 t, 2 r, 3 tr, 4 b, 5 bt, 6 br, 7 btr), in ascending order = the reference's order
__device__ double rs_cost_raw(const double *s1, const double *s2, double r, int *key);
__device__ double reedsshepp(const double *s1, const double *s2, double r, double s, Best &B) {
    const double dx = (s2[0] - s1[0]) / r, dy = (s2[1] - s1[1]) / r;
    double ct, st;
    sincos_(s1[2], &st, &ct);
    const double x0 = dx * ct + dy * st, y0 = -dx * st + dy * ct, t0 = mod2pi(s2[2] - s1[2]);
    double sb, cb;
    sincos_(t0, &sb, &cb);
    const double xb = x0 * cb + y0 * sb, yb = x0 * sb - y0 * cb;
    B.c = kInf; B.l = 0;
    for (int i = 0; i < 5; ++i) B.p[i] = mkseg(0, 0.0);
    // the sweep of simplecars.jl:283-339 keeps the first evaluation that attains the minimum; rs_cost_raw finds it
    // (cost + position in the sweep) with the shared-subexpression pass, and only that one is rebuilt with its control
    int key;
    rs_cost_raw(s1, s2, r, &key);
    const int fam = key >> 3, post = key & 7;
    {
        const int tr = post;
        const double bx = (tr & 4) ? xb : x0, by = (tr & 4) ? yb : y0;
        // timeflip: (-x, y, -th); reflect: (x, -y, -th)
        const double tx = (tr & 1) ? -bx : bx;
        const double ty = (tr & 2) ? -by : by;
        const bool neg = ((tr & 1) != 0) != ((tr & 2) != 0);
        rs_family(fam, tx, ty, neg ? -t0 : t0, neg ? -sb : sb, cb, B);
    }
    scale_segments(B, r, s);
    const int l = B.l;
    if (post & 1) for (int i = 0; i < l; ++i) B.p[i].u1 = -B.p[i].u1;
    if (post & 2) for (int i = 0; i < l; ++i) B.p[i].u2 = -B.p[i].u2;
    if (post & 4)
        for (int i = 0; i < l / 2; ++i) { const Seg tmp = B.p[i]; B.p[i] = B.p[l - 1 - i]; B.p[l - 1 - i] = tmp; }
    return B.c * r;
}

// ---- cost only (the table build needs no control): the same candidate lengths, evaluated target by target so that
// everything the families of one transformed target have in common -- sincos(tt), the polar form of (E, N), the
// acos of the C|C|C families -- is computed once.  The minimum of a set does not depend on the order it is taken in,
// so the result is the cost of reedsshepp() bit for bit.
// *key = 8 * family + target of the FIRST evaluation (in the reference's family-major order) that attains the
// minimum: the one whose control reedsshepp() returns
__device__ double rs_cost_raw(const double *s1, const double *s2, double r, int *key) {
    const double dx = (s2[0] - s1[0]) / r, dy = (s2[1] - s1[1]) / r;
    double ct, st;
    sincos_(s1[2], &st, &ct);
    const double x0 = dx * ct + dy * st, y0 = -dx * st + dy * ct, t0 = mod2pi(s2[2] - s1[2]);
    double sb, cb;
    sincos_(t0, &sb, &cb);
    const double xb = x0 * cb + y0 * sb, yb = x0 * sb - y0 * cb;
    double best = kInf;
    int best_key = 1 << 30;
#define MPB_TAKE(fam_, c_) do { const double c__ = (c_); const int k__ = 8 * (fam_) + tr;                \
        if (!(best <= c__) || (c__ == best && k__ < best_key)) { best = c__; best_key = k__; } } while (0)
#pragma unroll 1
    for (int tr = 0; tr < 8; ++tr) {
        const double bx = (tr & 4) ? xb : x0, by = (tr & 4) ? yb : y0;
        const double tx = (tr & 1) ? -bx : bx;
        const double ty = (tr & 2) ? -by : by;
        const bool neg = ((tr & 1) != 0) != ((tr & 2) != 0);
        const double tt = neg ? -t0 : t0, stt = neg ? -sb : sb, ctt = cb;
        const bool four = tr < 4;  // families tried on the first four targets only
        if (four) {
            {   // LpSpLp
                double rr, th;
                Rpolar(tx - stt, ty - 1.0 + ctt, &rr, &th);
                const double t = mod2pi(th), v = mod2pi(tt - t);
                MPB_TAKE(0, t + rr + v);
            }
            {   // LpSpRp
                double rr, th;
                Rpolar(tx + stt, ty - 1.0 - ctt, &rr, &th);
                if (!(rr * rr < 4.0)) {
                    const double u = sqrt(rr * rr - 4.0);
                    const double th1 = atan2_(2.0, u);
                    const double t = mod2pi(th + th1), v = mod2pi(t - tt);
                    MPB_TAKE(1, t + u + v);
                }
            }
        }
        {   // E = tx - sin, N = ty + cos - 1: LpRmLp (targets 0, 2), LpRmLm, LpRmSmLm
            const double E = tx - stt, N = ty + ctt - 1.0;
            const double EN = E * E + N * N;
            const double D = sqrt(EN), th = atan2_(N, E);
            if (!(EN > 16.0)) {
                double u = acos_(1.0 - D * D / 8.0);
                const double t = mod2pi(th - u / 2.0 + kPi);
                const double vv = mod2pi(kPi - u / 2.0 - th + tt);
                u = -u;
                if (tr == 0 || tr == 2) MPB_TAKE(2, t - u + vv);
                const double v3 = vv - kTwoPi;
                MPB_TAKE(3, t - u - v3);
            }
            if (!(D < 2.0)) {
                const double gamma = acos_(2.0 / D);
                const double F = sqrt(D * D / 4.0 - 1.0);
                const double t = mod2pi(kPi + th - gamma);
                const double u = 2.0 - 2.0 * F;
                if (!(u > 0.0)) {
                    const double v = mod2pi(-3.0 * kPi / 2.0 + gamma + tt - th) - kTwoPi;
                    MPB_TAKE(6, t + kPi / 2.0 - u - v);
                }
            }
        }
        {   // E = tx + sin, N = ty - cos - 1: LpRpuLmuRm, LpRmuLmuRp, LpRmSmLmRp (first four targets), LpRmSmRm (all)
            const double E = tx + stt, N = ty - ctt - 1.0;
            const double D = sqrt(E * E + N * N);
            if (four) {
                const double p = (2.0 + D) / 4.0;
                if (!(p < 0.0 || p > 1.0)) {
                    const double u = acos_(p);
                    double su, cu;
                    sincos_(u, &su, &cu);
                    const double tau = Tau(u, -u, E, N, su, cu);
                    const double t = mod2pi(tau);
                    const double v = mod2pi(Mwrap(tau - u + (-u) - tt)) - kTwoPi;
                    MPB_TAKE(4, t + 2.0 * u - v);
                }
                const double p2 = (20.0 - E * E - N * N) / 16.0;
                if (!(p2 < 0.0 || p2 > 1.0)) {
                    const double u = -acos_(p2);
                    double su, cu;
                    sincos_(u, &su, &cu);
                    const double tau = Tau(u, u, E, N, su, cu);
                    const double t = mod2pi(tau);
                    const double v = mod2pi(Mwrap(tau - u + u - tt));
                    MPB_TAKE(5, t - 2.0 * u + v);
                }
            }
            if (!(D < 2.0)) {
                const double beta = atan2_(N, E);
                {
                    const double t = mod2pi(beta + kPi / 2.0);
                    const double u = 2.0 - D;
                    if (!(u > 0.0)) {
                        const double v = mod2pi(-kPi - tt + beta) - kTwoPi;
                        MPB_TAKE(7, t + kPi / 2.0 - u - v);
                    }
                }
                if (four) {
                    const double gamma = acos_(2.0 / D);
                    const double F = sqrt(D * D / 4.0 - 1.0);
                    const double t = mod2pi(kPi + beta - gamma);
                    const double u = 4.0 - 2.0 * F;
                    if (!(u > 0.0)) {
                        const double v = mod2pi(kPi + beta - tt - gamma);
                        MPB_TAKE(8, t + kPi - u + v);
                    }
                }
            }
        }
    }
#undef MPB_TAKE
    *key = best_key;
    return best;
}
__device__ __forceinline__ double rs_cost(const double *s1, const double *s2, double r) {
    int key;
    return rs_cost_raw(s1, s2, r, &key) * r;
}

__device__ double dubins_cost(const double *s1, const double *s2, double r) {
    Best B;
    return dubins(s1, s2, r, 1.0, B);
}

__device__ __forceinline__ double steer(int kind, const double *v, const double *w, double rturn, double speed, Best &B) {
    return kind == MPB200_CAR_DUBINS ? dubins(v, w, rturn, speed, B) : reedsshepp(v, w, rturn, speed, B);
}

// evaluate(::ChoppedPreMetric, v, w) given the lower bound already computed (primitivetypes.jl:95-100)
__device__ __forceinline__ double chopped(int kind, double lb, const double *v, const double *w, double rturn, double chopval) {
    if (lb > chopval) return kInf;
    const double d = kind == MPB200_CAR_DUBINS ? dubins_cost(v, w, rturn) : rs_cost(v, w, rturn);
    return d <= chopval ? d : kInf;
}

// (s0, c0) = sincos(v[2])
__device__ __forceinline__ void propagate(const double *v, const Seg &u, double s0, double c0, double *out) {
    const double dth = u.t * u.u1 * u.u2;
    if (fabs(dth) > 10.0 * 2.220446049250313e-16) {
        double s1, c1;
        sincos_(v[2] + dth, &s1, &c1);
        out[0] = v[0] + (s1 - s0) / u.u2;
        out[1] = v[1] + (c0 - c1) / u.u2;
    } else {
        out[0] = v[0] + u.t * u.u1 * c0;
        out[1] = v[1] + u.t * u.u1 * s0;
    }
    out[2] = mod2pi(v[2] + dth);
}

template <int KIND>
__device__ __forceinline__ bool ws_free(const SpaceDev &S, const double *T, int M, const double *a, const double *b) {
    double p[2], q[2];
    state2workspace<3, 2>(S, a, p);
    state2workspace<3, 2>(S, b, q);
    if (KIND == 0) return !line_colliding_2d(T, p[0], p[1], q[0], q[1]);
    return box_segment_free<2>(T, M, p, q);
}

// is_free_motion(v, w, CC, SS): every waypoint but the last is bounds-checked, every consecutive pair swept
template <int KIND>
__device__ bool motion_free(int kind, double rturn, double speed, const SpaceDev &S, const double *T, int M,
                            const double *v, const double *w, int *checks) {
    Best B;
    steer(kind, v, w, rturn, speed, B);
    const double thres = kPi / 12.0;
    double cur[3] = {v[0], v[1], v[2]}, prev[3] = {v[0], v[1], v[2]};
    bool have_prev = false;
    for (int k = 0; k < B.l; ++k) {
        const Seg u = B.p[k];
        // first waypoint of the segment: its start state
        if (have_prev) {
            if (!in_state_space<3>(S, prev)) return false;
            *checks += 1;
            if (!ws_free<KIND>(S, T, M, prev, cur)) return false;
        }
        prev[0] = cur[0]; prev[1] = cur[1]; prev[2] = cur[2];
        have_prev = true;
        const long long m = (long long)floor(u.t * u.u1 * u.u2 / thres);
        double s0, c0;
        sincos_(cur[2], &s0, &c0);
        for (long long i = 1; i <= m && i < 32; ++i) {
            const double ang = (double)i * thres;
            double pt[3], sa, ca;
            sincos_(cur[2] + ang, &sa, &ca);
            pt[0] = cur[0] + (sa - s0) / u.u2;
            pt[1] = cur[1] + (c0 - ca) / u.u2;
            pt[2] = mod2pi(cur[2] + ang);
            if (!in_state_space<3>(S, prev)) return false;
            *checks += 1;
            if (!ws_free<KIND>(S, T, M, prev, pt)) return false;
            prev[0] = pt[0]; prev[1] = pt[1]; prev[2] = pt[2];
        }
        double nxt[3];
        propagate(cur, u, s0, c0, nxt);
        cur[0] = nxt[0]; cur[1] = nxt[1]; cur[2] = nxt[2];
    }
    if (have_prev) {  // push!(wps, w)
        if (!in_state_space<3>(S, prev)) return false;
        *checks += 1;
        if (!ws_free<KIND>(S, T, M, prev, w)) return false;
    }
    return true;
}

}  // namespace car

// ---- kernels -------------------------------------------------------------------------------------------------
__global__ void extract_xy_kernel(const double *__restrict__ V3, int64_t N, double *__restrict__ V2) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        V2[2 * i] = V3[3 * i];
        V2[2 * i + 1] = V3[3 * i + 1];
    }
}

// column of entry e (0-based) in a 1-based colptr
__device__ __forceinline__ int64_t column_of(const int64_t *__restrict__ colptr, int64_t ncols, int64_t e) {
    int64_t lo = 0, hi = ncols;  // colptr[lo] - 1 <= e < colptr[hi] - 1
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (colptr[mid] - 1 <= e) lo = mid; else hi = mid;
    }
    return lo;
}

// pass A: one thread per candidate entry of the (x, y) r-ball table: chopped cost(s), per-column counts
__global__ void __launch_bounds__(128)
car_cost_kernel(const double *__restrict__ V, const int64_t *__restrict__ colptr, const int64_t *__restrict__ rowval,
                const double *__restrict__ lbval, int64_t ncols, int64_t col0, int64_t nnz, int kind, double rturn,
                double r, double chopval, double *__restrict__ costF, double *__restrict__ costB,
                int *__restrict__ cntF, int *__restrict__ cntB) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nnz) return;
    const int64_t c = column_of(colptr, ncols, e);
    const int64_t i = rowval[e] - 1, q = col0 + c;
    const double v[3] = {V[3 * q], V[3 * q + 1], V[3 * q + 2]};
    const double w[3] = {V[3 * i], V[3 * i + 1], V[3 * i + 2]};
    const double lb = lbval[e];
    double d = car::chopped(kind, lb, v, w, rturn, chopval);
    if (!(d <= r)) d = car::kInf;
    costF[e] = d;
    if (d <= r) atomicAdd(&cntF[c], 1);
    if (costB) {
        double db = car::chopped(kind, lb, w, v, rturn, chopval);
        if (!(db <= r)) db = car::kInf;
        costB[e] = db;
        if (db <= r) atomicAdd(&cntB[c], 1);
    }
}

// pass B: one warp per column, ordered compaction of the kept entries
__global__ void __launch_bounds__(256)
car_compact_kernel(const int64_t *__restrict__ colptr, const int64_t *__restrict__ rowval, const double *__restrict__ cost,
                   int64_t ncols, const int64_t *__restrict__ colptr_out, int64_t *__restrict__ rowval_out,
                   double *__restrict__ nzval_out) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t c = gw; c < ncols; c += nw) {
        const int64_t beg = colptr[c] - 1, end = colptr[c + 1] - 1;
        int64_t at = colptr_out[c] - 1;
        for (int64_t e0 = beg; e0 < end; e0 += 32) {
            const int64_t e = e0 + lane;
            const double d = e < end ? cost[e] : car::kInf;
            const bool keep = d < car::kInf;
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (keep) {
                const int64_t o = at + __popc(m & ((1u << lane) - 1u));
                rowval_out[o] = rowval[e];
                nzval_out[o] = d;
            }
            at += __popc(m);
        }
    }
}

__device__ __forceinline__ const double *stage_table(const double *__restrict__ g_table, int words, bool use_smem, double *smem) {
    if (!use_smem) return g_table;
    for (int i = threadIdx.x; i < words; i += blockDim.x) smem[i] = g_table[i];
    __syncthreads();
    return smem;
}

// one thread per stored entry (row y, column x): the motion V[y] -> V[x]; one validity word per warp
template <int KIND>
__global__ void __launch_bounds__(128)
car_edges_free_kernel(const double *__restrict__ V, const int64_t *__restrict__ colptr, const int64_t *__restrict__ rowval,
                      int64_t ncols, int64_t col0, int64_t nnz, int kind, double rturn, double speed, SpaceDev S,
                      const double *__restrict__ g_table, int table_words, int M, bool use_smem,
                      uint32_t *__restrict__ bits32, unsigned long long *__restrict__ checks) {
    extern __shared__ double s_table[];
    const double *T = stage_table(g_table, table_words, use_smem, s_table);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool ok = false;
    int nchk = 0;
    if (e < nnz) {
        const int64_t c = column_of(colptr, ncols, e);
        const int64_t y = rowval[e] - 1, x = col0 + c;
        const double a[3] = {V[3 * y], V[3 * y + 1], V[3 * y + 2]};
        const double b[3] = {V[3 * x], V[3 * x + 1], V[3 * x + 2]};
        ok = car::motion_free<KIND>(kind, rturn, speed, S, T, M, a, b, &nchk);
    }
    const unsigned m = __ballot_sync(0xffffffffu, ok);
    unsigned long long n = (unsigned long long)nchk;
#pragma unroll
    for (int o = 16; o; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
    if ((threadIdx.x & 31) == 0) {
        if (e < nnz) bits32[e >> 5] = m;
        if (n) atomicAdd(checks, n);
    }
}

template <int KIND>
__global__ void __launch_bounds__(128)
car_motions_free_kernel(const double *__restrict__ A, const double *__restrict__ Bv, int64_t n, int kind, double rturn,
                        double speed, SpaceDev S, const double *__restrict__ g_table, int table_words, int M, bool use_smem,
                        uint8_t *__restrict__ out, unsigned long long *__restrict__ checks) {
    extern __shared__ double s_table[];
    const double *T = stage_table(g_table, table_words, use_smem, s_table);
    unsigned long long mine = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double a[3] = {A[3 * i], A[3 * i + 1], A[3 * i + 2]};
        const double b[3] = {Bv[3 * i], Bv[3 * i + 1], Bv[3 * i + 2]};
        int nchk = 0;
        out[i] = car::motion_free<KIND>(kind, rturn, speed, S, T, M, a, b, &nchk) ? 1 : 0;
        mine += nchk;
    }
    if (mine) atomicAdd(checks, mine);
}

__global__ void __launch_bounds__(128)
car_steer_kernel(const double *__restrict__ A, const double *__restrict__ Bv, int64_t n, int kind, double rturn, double speed,
                 double *__restrict__ cost, int *__restrict__ nseg, double *__restrict__ segs) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double a[3] = {A[3 * i], A[3 * i + 1], A[3 * i + 2]};
        const double b[3] = {Bv[3 * i], Bv[3 * i + 1], Bv[3 * i + 2]};
        car::Best B;
        cost[i] = car::steer(kind, a, b, rturn, speed, B);
        nseg[i] = B.l;
        for (int k = 0; k < 5; ++k) {
            segs[15 * i + 3 * k] = k < B.l ? B.p[k].t : 0.0;
            segs[15 * i + 3 * k + 1] = k < B.l ? B.p[k].u1 : 0.0;
            segs[15 * i + 3 * k + 2] = k < B.l ? B.p[k].u2 : 0.0;
        }
    }
}

// ---- host side -------------------------------------------------------------------------------------------------
int make_space(const mpb200_space_desc *ss, int d_state, SpaceDev *out, int *dw);

int car_args(int32_t kind, double rturn, double speed) {
    MPB_CHECK_ARG(kind == MPB200_CAR_REEDS_SHEPP || kind == MPB200_CAR_DUBINS, "kind must be MPB200_CAR_REEDS_SHEPP or MPB200_CAR_DUBINS");
    MPB_CHECK_ARG(rturn > 0 && rturn < std::numeric_limits<double>::infinity(), "turning radius must be positive");
    MPB_CHECK_ARG(speed > 0 && speed < std::numeric_limits<double>::infinity(), "speed must be positive");
    return MPB200_OK;
}

int car_extract_xy_device(const double *dV3, int64_t N, double *dV2) {
    if (N == 0) return 0;
    const unsigned g = (unsigned)std::min<int64_t>(ceil_div(N, 256), (int64_t)ctx().sm_count * 8);
    extract_xy_kernel<<<g, 256, 0, ctx().stream>>>(dV3, N, dV2);
    MPB_LAUNCHED();
    return 0;
}

static int finish_table(mpb200_table *out, const mpb200_table *cand, const mpb200_samples *s, int *cnt, const double *cost,
                        double r, DevBuf &scan_tmp, int64_t *d_total, int64_t *h_total) {
    Context &c = ctx();
    cudaStream_t st = c.stream;
    const int64_t nc = cand->ncols;
    if (int rc = out->colptr.reserve(sizeof(int64_t) * (size_t)(nc + 1))) return rc;
    if (int rc = exclusive_scan<int, int64_t>(cnt, nc, out->colptr.as<int64_t>(), (int64_t)1, scan_tmp, d_total)) return rc;
    MPB_CUDA(cudaMemcpyAsync(h_total, d_total, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    MPB_CUDA(cudaStreamSynchronize(st));
    const int64_t nnz = *h_total;
    if (int rc = out->rowval.reserve(sizeof(int64_t) * (size_t)(nnz + 1))) return rc;
    if (int rc = out->nzval.reserve(sizeof(double) * (size_t)(nnz + 1))) return rc;
    if (nc > 0 && nnz > 0) {
        const unsigned g = (unsigned)std::min<int64_t>(ceil_div(nc, 8), (int64_t)c.sm_count * 8);
        car_compact_kernel<<<g, 256, 0, st>>>(cand->colptr.as<int64_t>(), cand->rowval.as<int64_t>(), cost, nc,
                                              out->colptr.as<int64_t>(), out->rowval.as<int64_t>(), out->nzval.as<double>());
        MPB_LAUNCHED();
    }
    out->nnz = nnz; out->ncols = nc; out->col0 = cand->col0; out->r = r; out->euclid = false;
    out->src_N = s->N; out->src_d = s->d; out->src_serial = s->serial; out->edge_bits_valid = false; out->has_order = false;
    return 0;
}

// cand: the Euclidean r-ball table over the (x, y) columns of s (same query range); tB == NULL for Reeds-Shepp
int car_inball_device(const mpb200_samples *s, const mpb200_table *cand, int kind, double rturn, double r, double chopval,
                      mpb200_table *tF, mpb200_table *tB, DevBuf &work, DevBuf &scan_tmp) {
    Context &c = ctx();
    cudaStream_t st = c.stream;
    const int64_t nc = cand->ncols, nnz = cand->nnz;
    const bool both = tB != nullptr;
    // work: costF | costB | cntF | cntB
    const size_t cost_bytes = sizeof(double) * (size_t)(nnz + 1), cnt_bytes = sizeof(int) * (size_t)(nc + 2);
    if (int rc = work.reserve((both ? 2 : 1) * cost_bytes + 2 * cnt_bytes + 64)) return rc;
    double *costF = work.as<double>();
    double *costB = both ? costF + (nnz + 1) : nullptr;
    int *cntF = reinterpret_cast<int *>(costF + (both ? 2 : 1) * (nnz + 1));
    int *cntB = cntF + (nc + 2);
    MPB_CUDA(cudaMemsetAsync(cntF, 0, 2 * cnt_bytes, st));
    phase_bank(MPB200_OP_TABLE);
    phase_mark(0);
    if (nnz > 0) {
        car_cost_kernel<<<(unsigned)ceil_div(nnz, 128), 128, 0, st>>>(
            s->V.as<double>(), cand->colptr.as<int64_t>(), cand->rowval.as<int64_t>(), cand->nzval.as<double>(), nc,
            cand->col0, nnz, kind, rturn, r, chopval, costF, costB, cntF, cntB);
        MPB_LAUNCHED();
    }
    phase_mark(1);
    if (int rc = finish_table(tF, cand, s, cntF, costF, r, scan_tmp, c.d_scalar, c.h_scalar)) return rc;
    if (both)
        if (int rc = finish_table(tB, cand, s, cntB, costB, r, scan_tmp, c.d_scalar + 1, c.h_scalar + 1)) return rc;
    phase_mark(2);
    phases_collect(2);
    return 0;
}

struct ObsLaunch { const double *table; int words, M; bool use_smem; size_t smem; };
static ObsLaunch obs_cfg(const mpb200_obstacles *o) {
    ObsLaunch C;
    C.table = o->table.as<double>();
    C.words = o->table_words;
    C.M = o->M;
    const size_t bytes = sizeof(double) * (size_t)o->table_words;
    C.use_smem = bytes <= 160 * 1024;
    C.smem = C.use_smem ? bytes : 0;
    return C;
}
static int car_space(const mpb200_obstacles *o, const mpb200_space_desc *ss, SpaceDev *S) {
    int dw = 0;
    if (int rc = make_space(ss, 3, S, &dw)) return rc;
    if (dw != 2) return fail(MPB200_EARG, "car spaces have a 2-D workspace (state2workspace = VectorView(1:2))");
    if (o->kind == 1 && o->d != 2) return fail(MPB200_EARG, "box dimension %d != workspace dimension 2", o->d);
    return 0;
}

int car_edges_free_device(const mpb200_samples *s, const mpb200_table *t, int kind, double rturn, double speed,
                          const mpb200_obstacles *o, const mpb200_space_desc *ss, uint32_t *d_bits32,
                          unsigned long long *d_checks) {
    SpaceDev S;
    if (int rc = car_space(o, ss, &S)) return rc;
    if (t->nnz == 0) return 0;
    const ObsLaunch C = obs_cfg(o);
    cudaStream_t st = ctx().stream;
    const unsigned grid = (unsigned)ceil_div(t->nnz, 128);
#define CALL(K_)                                                                                                       \
    do {                                                                                                               \
        if (C.smem > 48 * 1024)                                                                                        \
            MPB_CUDA(cudaFuncSetAttribute(car_edges_free_kernel<K_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C.smem)); \
        car_edges_free_kernel<K_><<<grid, 128, C.smem, st>>>(s->V.as<double>(), t->colptr.as<int64_t>(), t->rowval.as<int64_t>(), \
                                                             t->ncols, t->col0, t->nnz, kind, rturn, speed, S, C.table, C.words, \
                                                             C.M, C.use_smem, d_bits32, d_checks);                     \
    } while (0)
    if (o->kind == 0) CALL(0); else CALL(1);
#undef CALL
    MPB_LAUNCHED();
    return 0;
}

int car_motions_free_device(int kind, double rturn, double speed, const double *dA, const double *dB, int64_t n,
                            const mpb200_obstacles *o, const mpb200_space_desc *ss, uint8_t *d_out, unsigned long long *d_checks) {
    SpaceDev S;
    if (int rc = car_space(o, ss, &S)) return rc;
    const ObsLaunch C = obs_cfg(o);
    cudaStream_t st = ctx().stream;
    const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(n, 128), (int64_t)ctx().sm_count * 16);
#define CALL(K_)                                                                                                       \
    do {                                                                                                               \
        if (C.smem > 48 * 1024)                                                                                        \
            MPB_CUDA(cudaFuncSetAttribute(car_motions_free_kernel<K_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C.smem)); \
        car_motions_free_kernel<K_><<<grid, 128, C.smem, st>>>(dA, dB, n, kind, rturn, speed, S, C.table, C.words, C.M, \
                                                               C.use_smem, d_out, d_checks);                           \
    } while (0)
    if (o->kind == 0) CALL(0); else CALL(1);
#undef CALL
    MPB_LAUNCHED();
    return 0;
}

int car_steer_device(int kind, double rturn, double speed, const double *dA, const double *dB, int64_t n, double *d_cost,
                     int *d_nseg, double *d_segs) {
    const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(n, 128), (int64_t)ctx().sm_count * 16);
    car_steer_kernel<<<grid, 128, 0, ctx().stream>>>(dA, dB, n, kind, rturn, speed, d_cost, d_nseg, d_segs);
    MPB_LAUNCHED();
    return 0;
}

// lazy GMT*: step 4 runs the car motion check of car_edges_free_kernel on the winning entry, on one lane
template <int KIND>
struct GmtCarEdge {
    static constexpr bool kLazy = true;
    int kind;
    double rturn, speed;
    SpaceDev S;
    const double *T;
    int M;
    __device__ bool operator()(const GmtArgs &a, long long, int y, int x, GmtCtl *ctl) const {
        double v[3], w[3];
        gmt_endpoints<3>(a, y, x, v, w);
        int nchk = 0;
        const bool ok = car::motion_free<KIND>(kind, rturn, speed, S, T, M, v, w, &nchk);
        gmt_count_segments(ctl, nchk);
        return ok;
    }
};

int gmt_lazy_car(const GmtArgs &a, int kind, double rturn, double speed, const mpb200_obstacles *o,
                 const mpb200_space_desc *ss, int *blocks) {
    SpaceDev S;
    if (int rc = car_space(o, ss, &S)) return rc;
    if (o->kind == 0) return gmt_launch(a, GmtCarEdge<0>{kind, rturn, speed, S, o->table.as<double>(), o->M}, blocks);
    return gmt_launch(a, GmtCarEdge<1>{kind, rturn, speed, S, o->table.as<double>(), o->M}, blocks);
}

}  // namespace mpb
