// ORACLE — TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is shipped or measured as the
// product; only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
// legs may build, load or call it.
//
// Scalar arithmetic of the rs-sync loss engine, restated on the CPU.  Every function cites the
// reference lines it follows (paths relative to /root/reference).  The arithmetic contract
// ("the spec", DESIGN.md §3) is: IEEE-754 binary64, round-to-nearest, NO implicit contraction
// (build with -ffp-contract=off); a fused multiply-add happens exactly where fma() is written;
// sums over a frame's rays are taken in a fixed order (RaySum, rssync_oracle.cpp), sums over
// frames in double-double so their value does not depend on the order of the terms.  The CUDA kernels implement the same contract, which is what makes bit-level
// parity checks possible.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>

#include "log1p_table.hpp"

namespace orc {

// ---------------------------------------------------------------------------------------------
// fused multiply-add: hardware FMA when the translation unit is compiled for it (the hot
// functions are cloned for "fma" targets), libm's exact software fma otherwise.
static inline double fmad(double a, double b, double c) { return __builtin_fma(a, b, c); }

// ---------------------------------------------------------------------------------------------
// Order-independent summation (double-double accumulator).  Stands in for arma::accu / arma::sum
// / arma::norm's inner sum (core_private.cpp:79,85,122; inline_utils.hpp:32-36) whose summation
// order is Armadillo-version specific anyway.
struct DD {
    double hi = 0.0, lo = 0.0;
    inline void add(double x) {
        double s = hi + x;
        double bb = s - hi;
        double e = (hi - (s - bb)) + (x - bb);
        hi = s;
        lo += e;
    }
    inline void merge(const DD& o) {
        double s = hi + o.hi;
        double bb = s - hi;
        double e = (hi - (s - bb)) + (o.hi - bb);
        hi = s;
        lo = (lo + o.lo) + e;
    }
    inline double value() const { return hi + lo; }
};

// ---------------------------------------------------------------------------------------------
// log1p for x >= 0 (the only domain the engine uses: x = r*r, core_private.cpp:82,121,354;
// inline_utils.hpp:28-30).  The reference calls libm's log1p through arma::log1p; libm results
// are not reproducible across platforms, so the spec fixes a division-free table algorithm with a
// stated operation order:
//   u = 1 + x, c = x - (u - 1) (the rounding error of u, exact);  u = 2^k m, m in [1, 2);
//   i = top 8 mantissa bits of m, (invc, logc) = table[i] (invc ~ 1/centre of the interval,
//   logc = -log(invc); entry 0 is (1, 0) so that small x keep full relative accuracy);
//   r = fma(m, invc, -1), |r| <= 2^-8;  log1p(r) = r + r^2 Q(r) with the degree-7 Taylor series;
//   c/u ~ c invc (1 - r) 2^-k;  result = (k ln2_hi + logc) + (log1p(r) + (k ln2_lo + c/u)).
// Agreement with a 80-digit log1p is <= 2 ulp (tests/test_oracle_math.py).
static inline uint32_t hi_word(double x) {
    uint64_t b;
    std::memcpy(&b, &x, 8);
    return (uint32_t)(b >> 32);
}
static inline double with_hi_word(double x, uint32_t hw) {
    uint64_t b;
    std::memcpy(&b, &x, 8);
    b = (b & 0xffffffffULL) | ((uint64_t)hw << 32);
    double r;
    std::memcpy(&r, &b, 8);
    return r;
}

static inline double log1p_nonneg(double x) {
    const double ln2_hi = 6.93147180369123816490e-01;
    const double ln2_lo = 1.90821492927058770002e-10;
    const double C2 = -0.5, C3 = 1.0 / 3.0, C4 = -0.25, C5 = 0.2, C6 = -1.0 / 6.0, C7 = 1.0 / 7.0;
    if (!(x < std::numeric_limits<double>::infinity())) return x;  // +inf, NaN
    const double u = 1.0 + x;
    const double c = x - (u - 1.0);
    const uint32_t hu = hi_word(u);
    const int k = (int)(hu >> 20) - 1023;
    const uint32_t i = (hu >> 12) & 0xffu;
    const double m = with_hi_word(u, (hu & 0x000fffffu) | 0x3ff00000u);
    const double invc = kLog1pTable[2 * i], logc = kLog1pTable[2 * i + 1];
    const double r = fmad(m, invc, -1.0);
    double q = fmad(r, C7, C6);
    q = fmad(r, q, C5);
    q = fmad(r, q, C4);
    q = fmad(r, q, C3);
    q = fmad(r, q, C2);
    const double r2 = r * r;
    const double p = fmad(r2, q, r);
    double t = c * invc;
    t = fmad(-r, t, t);
    const double corr = t * with_hi_word(0.0, (uint32_t)(1023 - k) << 20);  // * 2^-k
    const double dk = (double)k;
    const double lo = fmad(dk, ln2_lo, corr);
    const double hi = fmad(dk, ln2_hi, logc);
    return hi + (p + lo);
}

// ---------------------------------------------------------------------------------------------
// Pinned counter-based RNG replacing mtrand (inline_utils.hpp:13-17), which is seeded from
// std::random_device per thread and therefore irreproducible.  SURVEY.md §8(c) "Pinned RNG
// spec": stateless hash of (seed, stream, call_no, offset_idx, frame_id, iter, k).
static inline uint64_t mix64(uint64_t z) {
    z ^= z >> 30;
    z *= 0xBF58476D1CE4E5B9ULL;
    z ^= z >> 27;
    z *= 0x94D049BB133111EBULL;
    z ^= z >> 31;
    return z;
}
enum RngStream : uint64_t { kStreamPreSync = 1, kStreamDebugPreSync = 2, kStreamSyncInit = 3 };

static inline uint64_t rng_task_key(uint64_t seed, uint64_t stream, uint64_t call_no,
                                    uint64_t offset_idx, int64_t frame_id) {
    uint64_t h = mix64(seed + 0x9E3779B97F4A7C15ULL);
    h = mix64(h ^ (stream + (call_no << 8)));
    h = mix64(h ^ offset_idx);
    h = mix64(h ^ (uint64_t)frame_id);
    return h;
}
// index in [0, n): high 64 bits of draw * n
static inline uint32_t rng_index(uint64_t task_key, uint32_t iter, uint32_t k, uint32_t n) {
    uint64_t d = mix64(task_key ^ (((uint64_t)iter << 32) | (uint64_t)k));
    return (uint32_t)(((unsigned __int128)d * (unsigned __int128)n) >> 64);
}

// ---------------------------------------------------------------------------------------------
// Natural cubic spline on unit-spaced knots: minispline.cpp:3-46 (set_points) and :48-55
// (operator()).  Coefficients are stored per knot as a 16-double record
// { y[4], b[4], c[4], d[4] } for the four quaternion components (ndspline.cpp:13-27).
static inline void spline_build_1d(const double* y, long n, long ystride, double* rec, int comp) {
    // rec layout: rec[i*16 + 0*4 + comp] = y, + 1*4 = b, + 2*4 = c, + 3*4 = d
    // tridiagonal rows [lo, di, up]; boundary rows [.,2,0] and [0,2,.] (minispline.cpp:7-20)
    double* lo = new double[n];
    double* di = new double[n];
    double* up = new double[n];
    double* c = new double[n];
    for (long i = 0; i < n; ++i) { lo[i] = 0.0; di[i] = 0.0; up[i] = 0.0; c[i] = 0.0; }
    for (long i = 1; i < n - 1; ++i) {
        lo[i] = 1.0 / 3.0;
        di[i] = 2.0 / 3.0 * 2.0;
        up[i] = 1.0 / 3.0;
        c[i] = (y[(i + 1) * ystride] - 2 * y[i * ystride]) + y[(i - 1) * ystride];
    }
    di[0] = 2.0; up[0] = 0.0; c[0] = 0.0;
    di[n - 1] = 2.0; lo[n - 1] = 0.0; c[n - 1] = 0.0;
    for (long i = 0; i < n - 2; ++i) {  // forward elimination, minispline.cpp:22-26
        double k = 1. / di[i] * lo[i + 1];
        lo[i + 1] -= di[i] * k;
        di[i + 1] -= up[i] * k;
        c[i + 1] -= c[i] * k;
    }
    for (long i = n - 1; i > 1; --i) {  // back elimination, minispline.cpp:28-32
        double k = 1. / di[i] * up[i - 1];
        di[i - 1] -= lo[i] * k;
        up[i - 1] -= di[i] * k;
        c[i - 1] -= c[i] * k;
    }
    for (long i = 0; i < n; ++i) c[i] /= di[i];  // :34
    for (long i = 0; i < n; ++i) {
        double yi = y[i * ystride];
        double b, d;
        if (i < n - 1) {  // :38-41
            d = 1.0 / 3.0 * (c[i + 1] - c[i]);
            b = (y[(i + 1) * ystride] - yi) - 1.0 / 3.0 * (2.0 * c[i] + c[i + 1]);
        } else {  // :43-44 (n >= 2)
            d = 0.0;
            double dm = rec[(n - 2) * 16 + 12 + comp], cm = c[n - 2], bm = rec[(n - 2) * 16 + 4 + comp];
            b = (3.0 * dm + 2.0 * cm) + bm;
        }
        rec[i * 16 + 0 + comp] = yi;
        rec[i * 16 + 4 + comp] = b;
        rec[i * 16 + 8 + comp] = c[i];
        rec[i * 16 + 12 + comp] = d;
    }
    delete[] lo; delete[] di; delete[] up; delete[] c;
}

// spline::operator() for all four components at once (minispline.cpp:48-55, ndspline.cpp:21-27).
// idx = clamp(floor(x), 0, n); h = x - idx; x<0 -> left linear branch; x>n-1 -> right branch with
// the reference's h = x - min(floor(x), n) quirk; interior -> Horner.  The two linear branches are
// the Horner form with d := 0 (fma(0,h,c) == c exactly), which is how it is written here.
static inline void spline_eval4(const double* rec, long n, double x, double out[4]) {
    double fl = std::floor(x);
    double idxf = fl < 0.0 ? 0.0 : (fl > (double)n ? (double)n : fl);
    double h = x - idxf;
    long r = (long)idxf;
    if (r > n - 1) r = n - 1;
    bool extrap = (x < idxf) || (x > (double)(n - 1));
    const double* p = rec + r * 16;
    for (int c = 0; c < 4; ++c) {
        double d = extrap ? 0.0 : p[12 + c];
        out[c] = fmad(fmad(fmad(d, h, p[8 + c]), h, p[4 + c]), h, p[c]);
    }
}

// ---------------------------------------------------------------------------------------------
// One row of the problem matrix (core_private.cpp:19-28): spline at both timestamps,
// de-rotation of both rays, cross product.  Mathematically identical to
//   normalise(spline) -> conj(a) (x) (0,ray) (x) a  -> ar x br        (quat.cpp:33-47)
// with the two quaternion normalisations folded into one division:
//   rot(conj(q/|q|), p) = [ (w^2-u.u) p + 2 (u.p) u - 2 w (u x p) ] / |q|^2.
static inline void derotate_unnormalised(const double q[4], const double p[3], double out[3],
                                         double& n2) {
    const double w = q[0], u0 = q[1], u1 = q[2], u2 = q[3];
    const double uu = fmad(u2, u2, fmad(u1, u1, u0 * u0));
    n2 = fmad(w, w, uu);
    const double e = fmad(w, w, -uu);
    const double up = fmad(u2, p[2], fmad(u1, p[1], u0 * p[0]));
    const double up2 = up + up;
    const double c0 = fmad(u1, p[2], -(u2 * p[1]));
    const double c1 = fmad(u2, p[0], -(u0 * p[2]));
    const double c2 = fmad(u0, p[1], -(u1 * p[0]));
    const double w2 = w + w;
    out[0] = fmad(e, p[0], fmad(up2, u0, -(w2 * c0)));
    out[1] = fmad(e, p[1], fmad(up2, u1, -(w2 * c1)));
    out[2] = fmad(e, p[2], fmad(up2, u2, -(w2 * c2)));
}

static inline void problem_row(const double* rec, long n, double q0, double sr, double delay,
                               double ts_a, double ts_b, const double ra[3], const double rb[3],
                               double row[3]) {
    const double xa = ((ts_a - q0) + delay) * sr;  // core_private.cpp:19
    const double xb = ((ts_b - q0) + delay) * sr;  // :20
    double qa[4], qb[4], ar[3], br[3], na, nb;
    spline_eval4(rec, n, xa, qa);
    spline_eval4(rec, n, xb, qb);
    derotate_unnormalised(qa, ra, ar, na);
    derotate_unnormalised(qb, rb, br, nb);
    const double s = 1.0 / (na * nb);
    row[0] = fmad(ar[1], br[2], -(ar[2] * br[1])) * s;
    row[1] = fmad(ar[2], br[0], -(ar[0] * br[2])) * s;
    row[2] = fmad(ar[0], br[1], -(ar[1] * br[0])) * s;
}

static inline double dot3(const double a[3], const double b[3]) {
    return fmad(a[2], b[2], fmad(a[1], b[1], a[0] * b[0]));
}

// one component x*y - p of the estimator's hypothesis cross product (core_private.cpp:45), p the
// rounded product of the other pair: exactly 0 where the reference's rounded products cancel
// (parallel rows: a duplicated ray gives the reference's zero hypothesis), fma(x, y, -p) otherwise.
static inline double hyp_cross_term(double x, double y, double p) {
    return (x * y == p) ? 0.0 : fmad(x, y, -p);
}

// safe_normalize (inline_utils.hpp:5-11): vectors with norm < 1e-12 are left unscaled.
static inline void safe_normalize3(const double v[3], double out[3]) {
    double nrm = std::sqrt(dot3(v, v));
    if (nrm < 1e-12) { out[0] = v[0]; out[1] = v[1]; out[2] = v[2]; return; }
    double inv = 1.0 / nrm;
    out[0] = v[0] * inv; out[1] = v[1] * inv; out[2] = v[2] * inv;
}

static inline double clamp_k(double k) {  // inline_utils.hpp:50, std::clamp semantics
    return (k < 1e1) ? 1e1 : ((1e3 < k) ? 1e3 : k);
}

}  // namespace orc
