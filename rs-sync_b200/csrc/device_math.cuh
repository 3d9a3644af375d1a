// Device-side arithmetic of the rs-sync loss engine for sm_100a.
//
// Arithmetic contract (DESIGN.md §3): IEEE-754 binary64, round-to-nearest, compiled with
// -fmad=false so that a fused multiply-add happens exactly where fma() is written; sums over
// a frame's rays are taken in a fixed order (warp_sum), sums over frames go through a
// double-double accumulator so their value does not depend on how frames are distributed.  Reference lines each function stands for are cited inline (paths
// relative to the rs-sync repository).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "rng.h"

namespace rs {

// ---- double-double accumulation: the sums over FRAMES (the mutex-guarded `cost +=` of
// core_private.cpp:84-85, 235-237, 248-249), whose value must not depend on how frames are spread
// over warps, blocks or GPUs ----------------------------------------------------------------------
struct DD {
    double hi, lo;
};
__device__ __forceinline__ DD dd_zero() { return DD{0.0, 0.0}; }
__device__ __forceinline__ void dd_add(DD& a, double x) {
    double s = a.hi + x;
    double bb = s - a.hi;
    double e = (a.hi - (s - bb)) + (x - bb);
    a.hi = s;
    a.lo += e;
}
__device__ __forceinline__ void dd_merge(DD& a, const DD& b) {
    double s = a.hi + b.hi;
    double bb = s - a.hi;
    double e = (a.hi - (s - bb)) + (b.hi - bb);
    a.hi = s;
    a.lo = (a.lo + b.lo) + e;
}
// butterfly over the warp; every lane ends with the same (hi, lo).  Out of line: one copy of the
// 5-step butterfly instead of one per call site (instruction-cache footprint).
__device__ __noinline__ double warp_dd_sum(DD a) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        DD b;
        b.hi = __shfl_xor_sync(0xffffffffu, a.hi, off);
        b.lo = __shfl_xor_sync(0xffffffffu, a.lo, off);
        dd_merge(a, b);
    }
    return a.hi + a.lo;
}

// ---- sums over the rays of one frame (arma::accu / arma::sum / arma::norm inner sums) ----------
// Contract: the frame's rays in storage order (sorted by (ts_a, caller index)); ray j is added to
// partial sum j % 32 -- lane l of the warp, which owns rays l, l + 32, ... and adds them in that
// order starting from 0.0 -- and the 32 partial sums are combined by this xor butterfly (strides 16,
// 8, 4, 2, 1; a + b == b + a, so every lane ends with the same value).  The oracle adds in the same
// order (RaySum).
__device__ __forceinline__ double warp_sum(double a) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) a = a + __shfl_xor_sync(0xffffffffu, a, off);
    return a;
}
template <int N>
__device__ __forceinline__ void warp_sum_n(double (&a)[N]) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        double b[N];
#pragma unroll
        for (int j = 0; j < N; ++j) b[j] = __shfl_xor_sync(0xffffffffu, a[j], off);
#pragma unroll
        for (int j = 0; j < N; ++j) a[j] = a[j] + b[j];
    }
}

// ---- log1p on x >= 0 (arma::log1p at core_private.cpp:82,121,354; inline_utils.hpp:28-30) ----
// Division-free table algorithm; the operation order is part of the contract (the CPU oracle
// evaluates the same expression tree on the same table, csrc/log1p_table.h):
//   u = 1 + x, c = x - (u - 1) (rounding error of u, exact);  u = 2^k m, m in [1, 2);
//   (invc, logc) = table[top 8 mantissa bits of m]  (entry 0 is (1, 0): full relative accuracy for
//   small x);  r = fma(m, invc, -1), |r| <= 2^-8;  log1p(r) = r + r^2 Q(r), degree-7 Taylor;
//   c/u ~ c invc (1 - r) 2^-k;  result = (k ln2_hi + logc) + (log1p(r) + (k ln2_lo + c/u)).
// `tab` is the block's shared-memory copy of the table (load_log1p_table).
__device__ const double kLog1pTableDev[512] = {
#define RS_LOG1P_TABLE_BODY
#include "log1p_table.h"
#undef RS_LOG1P_TABLE_BODY
};
constexpr int kLog1pTableBytes = 512 * 8;

__device__ __forceinline__ void load_log1p_table(double* smem_tab) {
    for (int i = threadIdx.x; i < 512; i += blockDim.x) smem_tab[i] = kLog1pTableDev[i];
    __syncthreads();
}

__device__ __forceinline__ double log1p_nonneg(double x, const double* __restrict__ tab) {
    const double ln2_hi = 6.93147180369123816490e-01;
    const double ln2_lo = 1.90821492927058770002e-10;
    const double C2 = -0.5, C3 = 1.0 / 3.0, C4 = -0.25, C5 = 0.2, C6 = -1.0 / 6.0, C7 = 1.0 / 7.0;
    const double u = 1.0 + x;
    const double c = x - (u - 1.0);
    const unsigned hu = (unsigned)__double2hiint(u);
    const int k = (int)(hu >> 20) - 1023;
    const double m = __hiloint2double((int)((hu & 0x000fffffu) | 0x3ff00000u), __double2loint(u));
    const double2 e = *reinterpret_cast<const double2*>(
        reinterpret_cast<const char*>(tab) + ((hu >> 8) & 0xff0u));  // 16 B * (top 8 mantissa bits)
    const double r = fma(m, e.x, -1.0);
    double q = fma(r, C7, C6);
    q = fma(r, q, C5);
    q = fma(r, q, C4);
    q = fma(r, q, C3);
    q = fma(r, q, C2);
    const double r2 = r * r;
    const double p = fma(r2, q, r);
    double t = c * e.x;
    t = fma(-r, t, t);
    const double corr = t * __hiloint2double((1023 - k) << 20, 0);  // * 2^-k
    const double dk = (double)k;
    const double lo = fma(dk, ln2_lo, corr);
    const double hi = fma(dk, ln2_hi, e.y);
    const double res = hi + (p + lo);
    return (x < __longlong_as_double(0x7ff0000000000000LL)) ? res : x;  // +inf, NaN
}

// ---- pinned counter-based RNG (replaces mtrand, inline_utils.hpp:13-17) ----------------------
__device__ __forceinline__ uint32_t rng_index(uint64_t task_key, uint32_t iter, uint32_t k,
                                              uint32_t n) {
    uint64_t d = mix64(task_key ^ (((uint64_t)iter << 32) | (uint64_t)k));
    return (uint32_t)__umul64hi(d, (uint64_t)n);
}

// ---- natural cubic spline on unit knots, 4 components (minispline.cpp:48-55, ndspline.cpp:21-27)
// rec: n records of 16 doubles {y[4], b[4], c[4], d[4]}, 128-byte aligned, groups swizzled (below).
// General form: clamps, the linear extrapolation on both sides and the reference's right-side
// quirk (idx = n for x >= n, so h restarts at 0).  Only reached when x leaves [0, n-1).
// Record layout: the four 32-byte groups {y[4]}, {b[4]}, {c[4]}, {d[4]} of record i are stored at
// group position g ^ (i & 3) inside the 128-byte record.  Lanes of a warp touch two or three
// CONSECUTIVE records (the rays of a frame are sorted by timestamp); with the plain layout the same
// group of different records falls into the same shared-memory banks (records are 128 bytes = all
// 32 banks apart) and every coefficient load is a 2-3-way bank conflict; with the swizzle the groups
// of up to four consecutive records sit in four different bank octets.
struct Quat4 {
    double w, x, y, z;
};
struct RecGroups {
    const double2 *y, *b, *c, *d;
};
// record: address of record r (128-byte aligned, so or-ing / xor-ing bits 5-6 selects the group)
__device__ __forceinline__ RecGroups rec_groups(const double* record, unsigned r) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(record) | ((r & 3u) << 5);
    RecGroups g;
    g.y = reinterpret_cast<const double2*>(a);
    g.b = reinterpret_cast<const double2*>(a ^ 32u);
    g.c = reinterpret_cast<const double2*>(a ^ 64u);
    g.d = reinterpret_cast<const double2*>(a ^ 96u);
    return g;
}
__device__ __noinline__ Quat4 spline_eval4_edges(const double* __restrict__ rec, int n, double x) {
    const double fl = floor(x);
    const double idxf = fl < 0.0 ? 0.0 : (fl > (double)n ? (double)n : fl);
    const double h = x - idxf;
    int r = (int)idxf;
    r = r > n - 1 ? n - 1 : r;
    const bool extrap = (x < idxf) || (x > (double)(n - 1));
    const RecGroups p = rec_groups(rec + (size_t)r * 16, (unsigned)r);
    const double2 y01 = __ldg(p.y), y23 = __ldg(p.y + 1);
    const double2 b01 = __ldg(p.b), b23 = __ldg(p.b + 1);
    const double2 c01 = __ldg(p.c), c23 = __ldg(p.c + 1);
    double2 d01 = __ldg(p.d), d23 = __ldg(p.d + 1);
    if (extrap) { d01.x = d01.y = d23.x = d23.y = 0.0; }
    Quat4 q;
    q.w = fma(fma(fma(d01.x, h, c01.x), h, b01.x), h, y01.x);
    q.x = fma(fma(fma(d01.y, h, c01.y), h, b01.y), h, y01.y);
    q.y = fma(fma(fma(d23.x, h, c23.x), h, b23.x), h, y23.x);
    q.z = fma(fma(fma(d23.y, h, c23.y), h, b23.y), h, y23.y);
    return q;
}
__device__ __forceinline__ void spline_eval4(const double* __restrict__ rec, int n, double x,
                                             double q[4]) {
    const int r = __double2int_rd(x);  // floor; saturates for huge |x|, 0 for NaN
    if ((unsigned)r >= (unsigned)(n - 1)) {  // x outside [0, n-1): edges (and NaN, which has r = 0
        const Quat4 e = spline_eval4_edges(rec, n, x);  // only when n = 1)
        q[0] = e.w; q[1] = e.x; q[2] = e.y; q[3] = e.z;
        return;
    }
    const double h = x - (double)r;
    const RecGroups p = rec_groups(rec + (size_t)r * 16, (unsigned)r);
    const double2 y01 = __ldg(p.y), y23 = __ldg(p.y + 1);
    const double2 b01 = __ldg(p.b), b23 = __ldg(p.b + 1);
    const double2 c01 = __ldg(p.c), c23 = __ldg(p.c + 1);
    const double2 d01 = __ldg(p.d), d23 = __ldg(p.d + 1);
    q[0] = fma(fma(fma(d01.x, h, c01.x), h, b01.x), h, y01.x);
    q[1] = fma(fma(fma(d01.y, h, c01.y), h, b01.y), h, y01.y);
    q[2] = fma(fma(fma(d23.x, h, c23.x), h, b23.x), h, y23.x);
    q[3] = fma(fma(fma(d23.y, h, c23.y), h, b23.y), h, y23.y);
}

__device__ __noinline__ Quat4 spline_eval4_cold(const double* __restrict__ rec, int n, double x) {
    double q[4];
    spline_eval4(rec, n, x, q);
    return Quat4{q[0], q[1], q[2], q[3]};
}

// ---- de-rotation by the conjugate of an un-normalised quaternion (quat.cpp:33-47) ------------
//   |q|^2 * rot(conj(q/|q|), p) = (w^2 - u.u) p + 2 (u.p) u - 2 w (u x p)
__device__ __forceinline__ void derotate_unnormalised(const double q[4], double p0, double p1,
                                                      double p2, double out[3], double& n2) {
    const double w = q[0], u0 = q[1], u1 = q[2], u2 = q[3];
    const double uu = fma(u2, u2, fma(u1, u1, u0 * u0));
    n2 = fma(w, w, uu);
    const double e = fma(w, w, -uu);
    const double up = fma(u2, p2, fma(u1, p1, u0 * p0));
    const double up2 = up + up;
    const double c0 = fma(u1, p2, -(u2 * p1));
    const double c1 = fma(u2, p0, -(u0 * p2));
    const double c2 = fma(u0, p1, -(u1 * p0));
    const double w2 = w + w;
    out[0] = fma(e, p0, fma(up2, u0, -(w2 * c0)));
    out[1] = fma(e, p1, fma(up2, u1, -(w2 * c1)));
    out[2] = fma(e, p2, fma(up2, u2, -(w2 * c2)));
}

// one row of opt_compute_problem (core_private.cpp:19-28)
__device__ __forceinline__ void problem_row(const double* __restrict__ rec, int n, double q0,
                                            double sr, double delay, double ts_a, double ts_b,
                                            double ax, double ay, double az, double bx, double by,
                                            double bz, double row[3]) {
    const double xa = ((ts_a - q0) + delay) * sr;
    const double xb = ((ts_b - q0) + delay) * sr;
    double qa[4], qb[4], ar[3], br[3], na, nb;
    spline_eval4(rec, n, xa, qa);
    spline_eval4(rec, n, xb, qb);
    derotate_unnormalised(qa, ax, ay, az, ar, na);
    derotate_unnormalised(qb, bx, by, bz, br, nb);
    const double s = 1.0 / (na * nb);
    row[0] = fma(ar[1], br[2], -(ar[2] * br[1])) * s;
    row[1] = fma(ar[2], br[0], -(ar[0] * br[2])) * s;
    row[2] = fma(ar[0], br[1], -(ar[1] * br[0])) * s;
}

__device__ __forceinline__ double dot3(double a0, double a1, double a2, double b0, double b1,
                                       double b2) {
    return fma(a2, b2, fma(a1, b1, a0 * b0));
}

// one component x*y - p of the estimator's hypothesis cross product (core_private.cpp:45), p the
// rounded product of the other pair: fma(x, y, -p), except that it is exactly 0 where the
// reference's rounded products cancel (x*y == p).  Two equal rows (a duplicated ray) then give the
// reference's zero hypothesis, whose quartile 0 wins and whose non-finite residuals are the
// reference's panic, instead of a direction made of the products' rounding errors.
__device__ __forceinline__ double hyp_cross_term(double x, double y, double p) {
    return (x * y == p) ? 0.0 : fma(x, y, -p);
}

// safe_normalize (inline_utils.hpp:5-11)
__device__ __forceinline__ void safe_normalize3(double v0, double v1, double v2, double out[3]) {
    const double nrm = sqrt(dot3(v0, v1, v2, v0, v1, v2));
    if (nrm < 1e-12) { out[0] = v0; out[1] = v1; out[2] = v2; return; }
    const double inv = 1.0 / nrm;
    out[0] = v0 * inv; out[1] = v1 * inv; out[2] = v2 * inv;
}

__device__ __forceinline__ double clamp_k(double k) {  // inline_utils.hpp:50
    return (k < 1e1) ? 1e1 : ((1e3 < k) ? 1e3 : k);
}

__device__ __forceinline__ bool is_finite(double x) {
    return (__double2hiint(x) & 0x7ff00000) != 0x7ff00000;
}

}  // namespace rs
