// sm_100a kernels of the rs-sync synchronisation loss engine.
//
// Decomposition: ONE WARP PER (delay, frame) TASK.  A frame carries N <= 512 rays; lane l owns
// rays l, l+32, ... ("slots").  A task runs in phases that each keep their working set where it
// is cheapest:
//   A  rows      ray tiles + the spline window (PreSync: staged in shared memory by TMA bulk
//                copies; Sync: global loads) -> rows of the problem matrix (opt_compute_problem,
//                core_private.cpp:15-32) -> the warp's slice of shared memory (binary64 rows, and
//                for the estimator an fp32 row-normalised copy); a run-time loop over slots so the
//                heavy body (2 spline evaluations, 2 de-rotations, 1 division) exists once in the
//                instruction stream.
//   B  hypotheses  lanes 0..19 each build one plane normal from two random rows
//   C  estimator  opt_guess_translational_motion (:34-59) as an fp32x2 tournament with a rigorous
//                error margin; comparisons it cannot call are settled in binary64
//   D  loss       robust loss of the winning normal, fixed-order warp sums (pre_sync body
//                :79-85 / FrameState::Loss :92-123).
// Cross-lane work is warp shuffles / REDUX only; the one block-level mechanism is the mbarrier
// pipeline that stages phase A's inputs (presync_kernel).
// Instruction fetch matters as much as FP64 issue here (the first version of this kernel, fully
// unrolled over slots, was 91 KB of SASS and stalled 40 % of the time on instruction fetch,
// profiles/r01_presync_v1.md; unrolling phase A by two still costs 12 %): heavy bodies are written
// once, cold paths are __noinline__.  The arithmetic contract is in device_math.cuh.
#include "engine.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <map>
#include <mutex>
#include <tuple>
#include <utility>
#include <vector>

#include "device_math.cuh"
#include "gyro_scan.h"

namespace rs {

namespace {

constexpr unsigned FULL = 0xffffffffu;

// RS_CHECKED builds (make lib OUT=... EXTRA=-DRS_CHECKED) carry device-side assertions on every index
// that addresses shared memory or the arena, on the staging protocol's counters and on the lengths of
// the data-dependent loops; a violated assertion traps (the launch fails, the C ABI returns
// RSSYNC_E_CUDA).  compute-sanitizer is not available on the GPU pool this engine is developed on,
// so the whole -m gpu test suite is run against such a build instead (profiles/r02_checked_build.md).
#ifdef RS_CHECKED
__device__ int* g_assert_slot = nullptr;  // mapped host memory: survives a launch that dies afterwards
#define RS_ASSERT(cond)                                                      \
    do {                                                                     \
        if (!(cond) && g_assert_slot) {                                      \
            atomicCAS_system(g_assert_slot, 0, __LINE__);                    \
            __threadfence_system();                                          \
        }                                                                    \
    } while (0)
#else
#define RS_ASSERT(cond) do { } while (0)
#endif
#ifndef RS_WPB
#define RS_WPB 8
#endif
#ifndef RS_MINB
#define RS_MINB 3
#endif
constexpr int kWarpsPerBlock = RS_WPB;

std::atomic<uint64_t> g_launches{0};

// per-warp shared-memory slice: the raw rows of the problem matrix, SoA [3][NP], in STORAGE order
// (rays are stored sorted by ts_a).  That is ALL a task keeps in shared memory: the estimator's fp32
// row-normalised copy lives in registers (load_normalised_rows32), the cold binary64 paths work from
// registers too.  (r01 kept the fp32 copy and the cold paths' scratch here as well: 8.4 KB per warp
// instead of 5.25 KB at N = 200, which is what left no room to double-buffer the staged inputs.)
struct WarpSmem {
    double* P;
    float* hyp;  // estimator kernels: the current batch of hypotheses in fp32, [3][32]
};
constexpr size_t kHypBytes = 3 * 32 * 4;
__host__ __device__ constexpr size_t warp_smem_bytes(int NP) { return (size_t)NP * 3 * 8 + kHypBytes; }
__device__ __forceinline__ WarpSmem warp_smem(unsigned char* base, int warp, int NP) {
    WarpSmem w;
    w.P = reinterpret_cast<double*>(base + (size_t)warp * warp_smem_bytes(NP));
    w.hyp = reinterpret_cast<float*>(w.P + 3 * NP);
    return w;
}

// safe_normalize of one row (inline_utils.hpp:5-11): 1/|row|, 1.0 where |row| < 1e-12
__device__ __forceinline__ double row_inv_norm(double r0, double r1, double r2) {
    const double nrm = sqrt(dot3(r0, r1, r2, r0, r1, r2));
    return (nrm < 1e-12) ? 1.0 : 1.0 / nrm;
}

// ------------------------------------------------------------------------------------------
// Phase A.  Rows of the problem matrix for the whole frame -> shared memory (storage order, which is
// also the summation order of the contract's sums over rays; the estimator's random draws go through
// the `pos` plane).  Entries past the frame's last ray, up to NP, are zero rows.
__device__ __forceinline__ void build_rows_smem(const DeviceData& dd, const FrameDesc& fd, double delay,
                                                int lane, const WarpSmem& w, int NP) {
    const int nslots = (fd.n + 31) >> 5;
    for (int s = 0; s < nslots; ++s) {
        const int i = s * 32 + lane;
        const double* t = dd.rays + ((size_t)fd.off + s * 32) * 8 + lane;  // tile [8 fields][32 rays]
        const double tsa = __ldg(t), tsb = __ldg(t + 32);
        const double ax = __ldg(t + 64), ay = __ldg(t + 96), az = __ldg(t + 128);
        const double bx = __ldg(t + 160), by = __ldg(t + 192), bz = __ldg(t + 224);
        double row[3];
        problem_row(dd.rec, dd.nq, dd.q0, dd.sr, delay, tsa, tsb, ax, ay, az, bx, by, bz, row);
        if (i >= fd.n) { row[0] = row[1] = row[2] = 0.0; }
        w.P[i] = row[0];
        w.P[NP + i] = row[1];
        w.P[2 * NP + i] = row[2];
    }
    for (int i = nslots * 32 + lane; i < NP; i += 32) {
        w.P[i] = 0.0;
        w.P[NP + i] = 0.0;
        w.P[2 * NP + i] = 0.0;
    }
    __syncwarp();
}

// out-of-line copy for kernels whose hot path is the staged variant below
__device__ __noinline__ void build_rows_global_cold(const DeviceData& dd, const FrameDesc& fd, double delay,
                                                    int lane, const WarpSmem& w, int NP) {
    build_rows_smem(dd, fd, delay, lane, w, NP);
}

// ---- TMA bulk copies + mbarrier (PTX, sm_90+) --------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned long long* bar, unsigned parity) {
    unsigned ok;
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0u;
}
// global -> shared bulk copy (bytes: multiple of 16, both addresses 16-byte aligned); completion is
// signalled on `bar` as transaction bytes
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, unsigned bytes,
                                            unsigned long long* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// Phase A of the PreSync grid kernel: same arithmetic as build_rows_smem, with the frame's ray
// tiles (sTiles) and the spline records [rec_first, rec_first + rec_cnt) (sRec) staged in shared
// memory by TMA.  The window is computed from the frame's timestamp bounds with a record of slack, so
// every evaluation lands inside it and 0 <= x < 2^31 holds; the loop body is therefore branch-free
// (both spline evaluations of a ray issue their sixteen loads together and their eight Horner chains
// interleave): floor(x) is x + 2^52 rounded down, whose low word is the record index and whose
// difference from 2^52 is the exact (double)floor(x) of the contract's h = x - floor(x).  An index
// outside the window is clamped and remembered; such a task (none has been observed) is recomputed
// through the general path.
__device__ __forceinline__ double2 lds_f64x2(uint32_t addr) {
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ void spline_eval4_staged(uint32_t sRecAddr, unsigned at, unsigned r, double h,
                                                    double q[4]) {
    // the staged copy keeps the global layout: record r's groups are swizzled by r & 3 (rec_groups,
    // device_math.cuh).  Explicit shared-space loads: address arithmetic with xor hides the address
    // space from the compiler, which would fall back to generic loads.
    const uint32_t ay = (sRecAddr + at * 128u) | ((r & 3u) << 5);
    const uint32_t ab = ay ^ 32u, ac = ay ^ 64u, ad = ay ^ 96u;
    const double2 y01 = lds_f64x2(ay), y23 = lds_f64x2(ay + 16u), b01 = lds_f64x2(ab), b23 = lds_f64x2(ab + 16u);
    const double2 c01 = lds_f64x2(ac), c23 = lds_f64x2(ac + 16u), d01 = lds_f64x2(ad), d23 = lds_f64x2(ad + 16u);
    q[0] = fma(fma(fma(d01.x, h, c01.x), h, b01.x), h, y01.x);
    q[1] = fma(fma(fma(d01.y, h, c01.y), h, b01.y), h, y01.y);
    q[2] = fma(fma(fma(d23.x, h, c23.x), h, b23.x), h, y23.x);
    q[3] = fma(fma(fma(d23.y, h, c23.y), h, b23.y), h, y23.y);
}
__device__ __forceinline__ void build_rows_staged(const DeviceData& dd, const FrameDesc& fd, double delay,
                                                  int lane, const WarpSmem& w, int NP,
                                                  const double* __restrict__ sTiles,
                                                  const double* __restrict__ sRec, int rec_first,
                                                  int rec_cnt) {
    const int nslots = (fd.n + 31) >> 5;
    const double kTwo52 = 4503599627370496.0;
    const uint32_t sRecAddr = smem_u32(sRec);
    for (int s = 0; s < nslots; ++s) {
        const int i = s * 32 + lane;
        const double* t = sTiles + s * 256 + lane;
        const double xa = ((t[0] - dd.q0) + delay) * dd.sr;   // core_private.cpp:19-20
        const double xb = ((t[32] - dd.q0) + delay) * dd.sr;
        const double fa = __dadd_rd(xa, kTwo52), fb = __dadd_rd(xb, kTwo52);
        // record index inside the staged window.  No clamp: x is a monotone function of the timestamp
        // and of the delay, roundings included, the frame's ts_lo / ts_hi bound every timestamp of
        // its tile and the window was cut from their images with a record of slack either side
        // (grid_stage_unit), so the index lies in [1, rec_cnt - 3].  RS_CHECKED builds verify it.
        const unsigned ia = (unsigned)(__double2loint(fa) - rec_first);
        const unsigned ib = (unsigned)(__double2loint(fb) - rec_first);
        RS_ASSERT(ia >= 1u && ib >= 1u && ia + 2u < (unsigned)rec_cnt && ib + 2u < (unsigned)rec_cnt && i < NP);
        double qa[4], qb[4], ar[3], br[3], na, nb;
        spline_eval4_staged(sRecAddr, ia, ia + (unsigned)rec_first, xa - (fa - kTwo52), qa);
        spline_eval4_staged(sRecAddr, ib, ib + (unsigned)rec_first, xb - (fb - kTwo52), qb);
        derotate_unnormalised(qa, t[64], t[96], t[128], ar, na);
        derotate_unnormalised(qb, t[160], t[192], t[224], br, nb);
        const double sc = 1.0 / (na * nb);
        w.P[i] = fma(ar[1], br[2], -(ar[2] * br[1])) * sc;
        w.P[NP + i] = fma(ar[2], br[0], -(ar[0] * br[2])) * sc;
        w.P[2 * NP + i] = fma(ar[0], br[1], -(ar[1] * br[0])) * sc;
    }
    // entries past the frame's last ray are zero rows: the tail of the last slot (its padding rays
    // were evaluated like any other) and the slots up to NP
    for (int i = fd.n + lane; i < NP; i += 32) {
        w.P[i] = 0.0;
        w.P[NP + i] = 0.0;
        w.P[2 * NP + i] = 0.0;
    }
    __syncwarp();
}

// one hypothesis of opt_guess_translational_motion: plane normal through two random rows
// (core_private.cpp:41-46).  The draws index the caller's ray order; `pos` maps to storage.
__device__ __forceinline__ void draw_hypothesis(const DeviceData& dd, const FrameDesc& fd,
                                                const double* sP, int NP, uint64_t key, uint32_t it,
                                                double v[3]) {
    const uint32_t a = rng_index(key, it, 0u, (uint32_t)fd.n);  // :42
    uint32_t b, kk = 1u;
    do { b = rng_index(key, it, kk++, (uint32_t)fd.n); } while (b == a);  // :43
    const int pa = __ldg(dd.pos + fd.off + a), pb = __ldg(dd.pos + fd.off + b);
    RS_ASSERT(a < (uint32_t)fd.n && b < (uint32_t)fd.n && (unsigned)pa < (unsigned)fd.n && (unsigned)pb < (unsigned)fd.n);
    const double a0 = sP[pa], a1 = sP[NP + pa], a2 = sP[2 * NP + pa];
    const double b0 = sP[pb], b1 = sP[NP + pb], b2 = sP[2 * NP + pb];
    // where the reference's two rounded products cancel (parallel rows: a duplicated ray) its
    // component is exactly 0, not the products' rounding error that fma leaves (hyp_cross_term)
    const double c0 = hyp_cross_term(a1, b2, a2 * b1);
    const double c1 = hyp_cross_term(a2, b0, a0 * b2);
    const double c2 = hyp_cross_term(a0, b1, a1 * b0);
    safe_normalize3(c0, c1, c2, v);  // :45-46
}

// ------------------------------------------------------------------------------------------
// k-th smallest hi word (0-based) among the warp's keys, by quickselect over a per-lane bitmask
// of still-active slots.  Returns H and, through cl / ce, count(h < H) and count(h == H).
template <int SLOTS>
__device__ __forceinline__ unsigned pick_slot(const unsigned (&h)[SLOTS], int sb) {  // h[sb], sb dynamic
    unsigned v = h[0];
#pragma unroll
    for (int s = 1; s < SLOTS; ++s) v = (sb == s) ? h[s] : v;
    return v;
}
template <int SLOTS>
__device__ __forceinline__ unsigned warp_select_hi(const unsigned (&h)[SLOTS], int kth, unsigned bound_hi,
                                                   int lane, int& cl, int& ce) {
    // Quickselect on VALUE bounds: the answer lies in [L, U).  Keys are < 2^31, so the sign bit of a
    // difference is the `<` predicate: two subtract + shift-add pairs per key count (h < pivot) and
    // (h <= pivot) over ALL keys, no per-lane bookkeeping.  The pivot is any key inside [L, U),
    // found by probing one 32-key batch (one slot of every lane) at a time, a different batch
    // first in each round.
    unsigned L = 0u, U = bound_hi + 1u;
    int round = 0;
    for (;;) {
        unsigned pv = 0u;
        for (int j = 0;; ++j) {
            int sb = round + j;
            sb -= (sb / SLOTS) * SLOTS;
            const unsigned cand = pick_slot<SLOTS>(h, sb);
            const unsigned bal = __ballot_sync(FULL, (cand - L) < (U - L));
            if (bal) {
                const int rot = (round * 7 + 3) & 31;
                const unsigned rb = __funnelshift_r(bal, bal, rot);
                pv = __shfl_sync(FULL, cand, (__ffs(rb) - 1 + rot) & 31);
                break;
            }
        }
        const unsigned pv1 = pv + 1u;
        unsigned c1 = 0, c2 = 0;
#pragma unroll
        for (int s = 0; s < SLOTS; ++s) {
            c1 += (h[s] - pv) >> 31;
            c2 += (h[s] - pv1) >> 31;
        }
        const unsigned packed = __reduce_add_sync(FULL, c1 | (c2 << 16));
        const int nl = (int)(packed & 0xffffu), nle = (int)(packed >> 16);
        if (kth < nl) {
            U = pv;
        } else if (kth < nle) {
            cl = nl;
            ce = nle - nl;
            return pv;
        } else {
            L = pv1;
        }
        ++round;
    }
}

// Exact estimator: opt_guess_translational_motion (core_private.cpp:34-59) in binary64, the
// arithmetic contract itself.  A hypothesis wins iff more than n/4 of its squared residuals lie
// below the best quartile so far (<=> `med < least_med`, :53); only then is its exact quartile
// selected.  Residual keys are compared as (hi word, lo word) pairs of the non-negative doubles,
// i.e. in exact double order.  Runs when the fp32 tournament below cannot certify its winner.
struct Vec3 {
    double x, y, z;
};
template <int SLOTS>
__device__ __noinline__ Vec3 warp_ransac_exact(const DeviceData& dd, const FrameDesc& fd,
                                               const WarpSmem& w, int iters, uint64_t key, int lane) {
    double M[3];
    constexpr int NP = SLOTS * 32;
    const int n = fd.n;
    const unsigned long long nanbits = 0x7ff8000000000000ULL;
    __syncwarp();
    double np[SLOTS][3];
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
        const int i = s * 32 + lane;
        const double p0 = w.P[i], p1 = w.P[NP + i], p2 = w.P[2 * NP + i];
        // padding entries get inv = NaN: their residuals sort above everything
        const double inv = (i < n) ? row_inv_norm(p0, p1, p2) : __longlong_as_double((long long)nanbits);
        np[s][0] = p0 * inv;  // :35-36
        np[s][1] = p1 * inv;
        np[s][2] = p2 * inv;
    }
    const int kth = n / 4;  // :52
    unsigned least_hi = 0x7ff00000u, least_lo = 1u;  // just above +inf
    M[0] = M[1] = M[2] = 0.0;
    for (int j0 = 0; j0 < iters; j0 += 32) {
        double v[3] = {0.0, 0.0, 0.0};
        if (j0 + lane < iters) draw_hypothesis(dd, fd, w.P, NP, key, (uint32_t)(j0 + lane), v);
        const int cnt = (iters - j0) < 32 ? (iters - j0) : 32;
        for (int t = 0; t < cnt; ++t) {
            const double vx = __shfl_sync(FULL, v[0], t);
            const double vy = __shfl_sync(FULL, v[1], t);
            const double vz = __shfl_sync(FULL, v[2], t);
            double r2[SLOTS];
            unsigned h[SLOTS];
            // hi words of r^2 (non-negative doubles, NaN = 0x7ff80000) are < 2^31, so the sign
            // bit of (h - least_hi) is the `<` predicate and a zero difference flags a tie
            unsigned below = 0, dmin = 0xffffffffu;
#pragma unroll
            for (int s = 0; s < SLOTS; ++s) {
                const double r = dot3(np[s][0], np[s][1], np[s][2], vx, vy, vz);  // :48
                r2[s] = r * r;                                                      // :49
                h[s] = (unsigned)__double2hiint(r2[s]) & 0x7fffffffu;
                const unsigned d = h[s] - least_hi;
                below += d >> 31;
                dmin = min(dmin, d);
            }
            const unsigned packed = __reduce_add_sync(FULL, below | ((dmin == 0u ? 1u : 0u) << 16));
            int nbelow = (int)(packed & 0xffffu);
            if (packed >> 16) {  // hi-word ties with the threshold: settle them on the lo word
                unsigned extra = 0;
#pragma unroll
                for (int s = 0; s < SLOTS; ++s)
                    extra += (h[s] == least_hi && (unsigned)__double2loint(r2[s]) < least_lo) ? 1u : 0u;
                nbelow += (int)__reduce_add_sync(FULL, extra);
            }
            if (nbelow > kth) {  // med < least_med: select the exact quartile
                int cl, ce;
                const unsigned H = warp_select_hi<SLOTS>(h, kth, least_hi, lane, cl, ce);
                // rank (kth - cl) among the ce keys whose hi word is H, ordered by lo word
                int rem = kth - cl;
                unsigned cur = 0u, lo_ans = 0u;
                for (;;) {
                    unsigned mn = 0xffffffffu, c = 0u;
#pragma unroll
                    for (int s = 0; s < SLOTS; ++s) {
                        const unsigned lo = (unsigned)__double2loint(r2[s]);
                        if (h[s] == H && lo >= cur) mn = min(mn, lo);
                    }
                    mn = __reduce_min_sync(FULL, mn);
#pragma unroll
                    for (int s = 0; s < SLOTS; ++s)
                        c += (h[s] == H && (unsigned)__double2loint(r2[s]) == mn) ? 1u : 0u;
                    c = __reduce_add_sync(FULL, c);
                    if (rem < (int)c) { lo_ans = mn; break; }
                    rem -= (int)c;
                    cur = mn + 1u;
                }
                least_hi = H;
                least_lo = lo_ans;
                M[0] = vx; M[1] = vy; M[2] = vz;
            }
        }
    }
    return Vec3{M[0], M[1], M[2]};
}

// Exact (binary64, the contract's arithmetic) quartile of the squared residuals of ONE hypothesis,
// returned as the bit pattern of the non-negative double (bit patterns order like the values).
// Used by the tournament below to settle a comparison that fp32 cannot call.
template <int SLOTS>
__device__ __noinline__ unsigned long long warp_exact_quartile(const WarpSmem& w, int n, int lane,
                                                               double vx, double vy, double vz) {
    constexpr int NP = SLOTS * 32;
    const unsigned long long nanbits = 0x7ff8000000000000ULL;
    double r2[SLOTS];
    unsigned h[SLOTS];
    __syncwarp();
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
        const int i = s * 32 + lane;
        const double p0 = w.P[i], p1 = w.P[NP + i], p2 = w.P[2 * NP + i];
        const double inv = (i < n) ? row_inv_norm(p0, p1, p2) : __longlong_as_double((long long)nanbits);
        const double r = dot3(p0 * inv, p1 * inv, p2 * inv, vx, vy, vz);  // :35-36, :48
        r2[s] = r * r;                                                    // :49
        h[s] = (unsigned)__double2hiint(r2[s]) & 0x7fffffffu;
    }
    const int kth = n / 4;  // :52
    int cl, ce;
    const unsigned H = warp_select_hi<SLOTS>(h, kth, 0x7ff80000u, lane, cl, ce);
    int rem = kth - cl;  // rank among the ce keys whose hi word is H, ordered by lo word
    unsigned cur = 0u, lo_ans = 0u;
    for (;;) {
        unsigned mn = 0xffffffffu, c = 0u;
#pragma unroll
        for (int s = 0; s < SLOTS; ++s) {
            const unsigned lo = (unsigned)__double2loint(r2[s]);
            if (h[s] == H && lo >= cur) mn = min(mn, lo);
        }
        mn = __reduce_min_sync(FULL, mn);
#pragma unroll
        for (int s = 0; s < SLOTS; ++s)
            c += (h[s] == H && (unsigned)__double2loint(r2[s]) == mn) ? 1u : 0u;
        c = __reduce_add_sync(FULL, c);
        if (rem < (int)c) { lo_ans = mn; break; }
        rem -= (int)c;
        cur = mn + 1u;
    }
    return ((unsigned long long)H << 32) | lo_ans;
}

// ------------------------------------------------------------------------------------------
// fp32 tournament (the estimator's fast path).
//
// Only the ARGMIN over hypotheses of the quartile of the squared residuals matters (the first
// hypothesis with the strictly smallest quartile wins, core_private.cpp:53-56), never the quartile
// itself.  Let np, v, r = np.v be the contract's binary64 normalised row, hypothesis and residual
// (|np|, |v| <= 1).  The tournament uses a = fl32(row) * rsqrt.approx(fl32(|row|^2)), i.e.
// a_i = np_i (1 + e) with |e| <= (1/2 + 4 + 1 + 1) 2^-24 (conversion of |row|^2 halved by the square
// root, rsqrt.approx <= 2^-22, conversion of the row, product), w = fl32(v) and the fp32 fma chain
// rho (3 roundings): |rho - r| <= (6.5 + 1 + 3) 2^-24, and s = fl32(rho^2) has
// |sqrt(s) - |r|| <= kDelta = 11 * 2^-24 = 6.6e-7.  Order statistics are 1-Lipschitz in the sup
// norm, so the fp32 quartile q32 and the exact one q64 of a hypothesis satisfy
// |sqrt(q32) - sqrt(q64)| <= kDelta.  Hence, with up(x) >= (sqrt(x) + kMargin)^2 (directed
// rounding) and kMargin >= 2 kDelta:
//   * count(s_t <= up(q32_best)) <= n/4   =>  q64_t > q64_best        (t is rigorously worse)
//   * up(q32_t) < q32_best                =>  q64_t < q64_best        (t is rigorously better)
// Anything else is too close to call in fp32: that one comparison is settled with the exact
// binary64 quartiles of the two hypotheses (warp_exact_quartile; ties keep the earlier one), so the
// winner is always the exact estimator's M, bit for bit.  Only non-finite data sends the whole
// task to warp_ransac_exact.
constexpr float kMargin = 1.4e-6f;

__device__ __forceinline__ unsigned up_bits(unsigned qbits) {  // rigorous upper bound (directed rounding)
    const float u = __fadd_ru(__fsqrt_ru(__uint_as_float(qbits)), kMargin);
    return __float_as_uint(__fmul_ru(u, u));
}
__device__ __forceinline__ float sqrt_approx(float x) {
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// ---- order statistics over the warp's keys: SLOTS non-negative floats per lane, compared through
// their bit patterns --------------------------------------------------------------------------------
// count of keys <= pv (s <= pv  <=>  s - next(pv) < 0)
template <int SLOTS>
__device__ __forceinline__ int warp_count_le(const float (&s)[SLOTS], unsigned pv) {
    const float nt = -__uint_as_float(pv + 1u);
    unsigned c = 0;
#pragma unroll
    for (int i = 0; i < SLOTS; ++i) c += __float_as_uint(s[i] + nt) >> 31;
    return (int)__reduce_add_sync(FULL, c);
}
// smallest key >= lo (at least one exists)
template <int SLOTS>
__device__ __forceinline__ unsigned warp_min_ge(const float (&s)[SLOTS], unsigned lo) {
    unsigned mn = 0xffffffffu;
#pragma unroll
    for (int i = 0; i < SLOTS; ++i) mn = min(mn, __float_as_uint(s[i]) - lo);  // keys below lo wrap to >= 2^31
    return lo + __reduce_min_sync(FULL, mn);
}
// largest key < hi_excl (at least one exists)
template <int SLOTS>
__device__ __forceinline__ unsigned warp_max_lt(const float (&s)[SLOTS], unsigned hi_excl) {
    unsigned mn = 0xffffffffu;
    const unsigned top = hi_excl - 1u;
#pragma unroll
    for (int i = 0; i < SLOTS; ++i) mn = min(mn, top - __float_as_uint(s[i]));  // keys >= hi_excl wrap
    return top - __reduce_min_sync(FULL, mn);
}

// kk-th smallest (0-based) of the warp's SLOTS*32 keys, given count(key < hi_excl) = chi > kk.
// Value-bracket search [lo, hi_excl) with clo = count(key < lo) <= kk < chi.  Pivots: with no scale
// information (`sample`), the matching order statistic of a 32-key sample (slot 0 of every lane);
// afterwards interpolation in the sqrt domain (ranks of small residuals grow linearly in |r|),
// bisection of the bit pattern after two steps of poor progress.  When the wanted key is the
// lowest or highest of the bracket it is extracted with one warp min.
template <int SLOTS>
__device__ __forceinline__ unsigned warp_select32(const float (&s)[SLOTS], int kk, unsigned hi_excl,
                                                  int chi, int npad, int n, bool sample) {
    unsigned lo = 0u;
    int clo = 0, poor = 0;
    for (int round = 0;; ++round) {
        RS_ASSERT(round < 80 && clo <= kk && kk < chi && lo < hi_excl);  // bisection alone ends within 2 x 32 rounds
        if (hi_excl - lo == 1u) return lo;
        if (kk == clo) return warp_min_ge<SLOTS>(s, lo);
        if (kk == chi - 1) return warp_max_lt<SLOTS>(s, hi_excl);
        unsigned pv;
        if (sample) {
            sample = false;
            const int js = min((32 * (kk - npad)) / n, 31);
            const unsigned k0 = __float_as_uint(s[0]);
            unsigned cur = 0u;
            pv = 0u;
            for (int i = 0; i <= js; ++i) {
                pv = cur + __reduce_min_sync(FULL, k0 - cur);
                cur = pv + 1u;
            }
        } else if (poor >= 2) {
            poor = 0;
            pv = lo + ((hi_excl - lo) >> 1);
        } else {
            const int cl = (lo == 0u) ? npad : clo;  // the padding keys sit at +0
            const float frac = ((float)(kk - cl) + 0.5f) / (float)(chi - cl);
            const float sl = sqrt_approx(__uint_as_float(lo));
            const float sh = sqrt_approx(__uint_as_float(hi_excl));
            const float sq = fmaf(sh - sl, frac, sl);
            pv = __float_as_uint(sq * sq);
        }
        pv = max(pv, lo);
        pv = min(pv, hi_excl - 2u);
        const int cnt = warp_count_le<SLOTS>(s, pv);
        if (cnt > kk) {
            poor = (2 * (cnt - clo) > (chi - clo)) ? poor + 1 : 0;
            hi_excl = pv + 1u;
            chi = cnt;
        } else {
            poor = (2 * (chi - cnt) > (chi - clo)) ? poor + 1 : 0;
            lo = pv + 1u;
            clo = cnt;
        }
    }
}

// The tournament's inputs: the frame's rows, row-normalised, in fp32, in registers -- lane l holds
// the three components of its SLOTS rays.  Any accuracy the margin covers will do, so the norm is
// taken with rsqrt.approx (rel. error <= 2^-22.4).  Rows that safe_normalize would leave unscaled
// (|row| < 1e-12, also out of fp32 range) and non-finite rows poison `fin`.  fp32(1e-24) is above
// 1e-24, and |row|^2 just below 1e-24 rounds to it: hence <=, so that every row safe_normalize leaves
// unscaled is caught (a few just above 1e-12 are too, harmlessly): returns false, and the
// task goes to the exact estimator (which of the two it was is only worked out there, on the cold
// path: warp_ransac).  Rows past the frame's last ray (zero rows) become +0 keys.
template <int SLOTS>
__device__ __forceinline__ bool load_normalised_rows32(const double* __restrict__ sP, int n, int lane,
                                                       float (&nx)[SLOTS], float (&ny)[SLOTS],
                                                       float (&nz)[SLOTS]) {
    constexpr int NP = SLOTS * 32;
    float fin = 0.f;  // stays finite iff every row is (rows and 1/|row| feed it)
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
        const int i = s * 32 + lane;
        const double r0 = sP[i], r1 = sP[NP + i], r2 = sP[2 * NP + i];
        const float n2 = (float)dot3(r0, r1, r2, r0, r1, r2);
        float rs;
        asm("rsqrt.approx.f32 %0, %1;" : "=f"(rs) : "f"(n2));
        if (i >= n) rs = 0.f;
        else if (n2 <= 1e-24f) rs = __uint_as_float(0x7fc00000u);
        nx[s] = (float)r0 * rs;
        ny[s] = (float)r1 * rs;
        nz[s] = (float)r2 * rs;
        fin += (fabsf(nx[s]) + fabsf(ny[s])) + fabsf(nz[s]);  // non-finite row -> NaN
    }
    return __all_sync(FULL, (__float_as_uint(fin) & 0x7f800000u) != 0x7f800000u);
}

// Result of the fast path: the winner is certified / it is not (run the exact estimator) / a row is
// not finite or too small to normalise in fp32 (exact estimator; pre_sync's "non-finite numbers in P"
// condition only if a row component really is non-finite).
// kFastRetry: the run started from a prior threshold that turned out too tight (see `prior`): run again
// without one.
enum FastStatus { kFastOk = 0, kFastUndecided = 1, kFastRowsNotFinite = 2, kFastRetry = 3 };

// The tournament proper.  Hypotheses are taken two at a time: the packed fp32x2 instructions carry
// hypotheses t and t + 1 in their two halves against ONE ray (scalar operand), so a pass over the
// lane's SLOTS rays costs four packed instructions and two shift-adds per ray for two hypotheses,
// with one warp reduction for both counts.  (r01 packed two RAYS against one hypothesis: a pass per
// hypothesis over pairs_for(NP) ray pairs -- eight slots' worth of work for N = 200's seven -- and a
// reduction each.)  Both counts are against the threshold of the best hypothesis so far:
//   * both <= kk: both rigorously worse, next pair (the common case);
//   * the first has more: it is a challenger -- select its quartile, compare, maybe a new best --
//     and the second is looked at again, as the first of the next pair, against whatever the
//     threshold is then;
//   * only the second: the first is rejected, the threshold unchanged, the second is the challenger.
// The rejection test is made on the EXACT squares: e = fma(rho, rho, -thr1) is the correctly rounded
// rho^2 - thr1, whose sign is that of the exact difference, so the count is count(rho^2 < thr1);
// |rho| is at least as close to |r64| as sqrt(fl(rho^2)) is, so the argument at the top of this
// section holds for these keys as it does for the rounded ones.  A challenger's keys are the rounded
// squares (the select works on their bit patterns); its count is retaken on those -- it can differ
// where rho^2 rounds up to thr1, and is then just as rigorous a rejection.
// `hyp`: 3 x 32 floats of the warp's shared memory (the batch's hypotheses in fp32, by component).
//
// `prior` (0: none): a threshold to START from instead of the first hypothesis' quartile -- the grid
// kernel passes twice the winning quartile of the neighbouring delay of the same frame.  It acts as a
// best hypothesis that nobody holds: everything whose count below it does not exceed kk is rejected
// at once, exactly as against a real best (its exact rho^2 quartile is >= prior), and the first
// hypothesis that passes becomes the real best if its quartile is rigorously below the prior
// (up(q) < prior) -- then every earlier rejection also holds against it, because thr1 only went down.
// The sequential tournament raises its threshold-to-beat from nothing, so early hypotheses of median
// quality all pay for a select (3.6 selects per task on C2); from a good prior only hypotheses near
// the best do (2.3).  If nothing passes, or the first one that does is too close to the prior to
// call, the prior was too tight: kFastRetry, and the caller runs the plain tournament.  *tau_out:
// the winner's fp32 quartile (the next task's prior).
template <int SLOTS>
__device__ __forceinline__ FastStatus warp_ransac_fast(const DeviceData& dd, const FrameDesc& fd,
                                                       const WarpSmem& w, int iters, uint64_t key,
                                                       int lane, double M[3], int* settled,
                                                       unsigned prior, unsigned* tau_out) {
    constexpr int NP = SLOTS * 32;
    float nx[SLOTS], ny[SLOTS], nz[SLOTS];
    if (!load_normalised_rows32<SLOTS>(w.P, fd.n, lane, nx, ny, nz)) return kFastRowsNotFinite;
    const int n = fd.n;
    const int npad = NP - n;      // padding keys are +0: always counted, always below
    const int kk = n / 4 + npad;  // :52
    unsigned tau = 0x7f800000u;   // fp32 quartile of the best hypothesis so far (+inf: none yet)
    float nthr = 0.f;             // -thr1
    unsigned thr1 = 0u;           // nextafter(up(tau)): s <= up(tau)  <=>  s < thr1
    bool has_real = true;         // false while `tau` is the prior and no hypothesis holds it
    if (prior) {
        tau = thr1 = prior;
        nthr = -__uint_as_float(prior);
        has_real = false;
    }
    M[0] = M[1] = M[2] = 0.0;
    float* hyp = w.hyp;
    for (int j0 = 0; j0 < iters; j0 += 32) {
        double v[3] = {0.0, 0.0, 0.0};
        if (j0 + lane < iters) draw_hypothesis(dd, fd, w.P, NP, key, (uint32_t)(j0 + lane), v);
        __syncwarp();
        hyp[lane] = (float)v[0];
        hyp[32 + lane] = (float)v[1];
        hyp[64 + lane] = (float)v[2];
        __syncwarp();
        const int cnt = (iters - j0) < 32 ? (iters - j0) : 32;
        int t = 0;
        while (t < cnt) {
            float sq[SLOTS];  // keys of the hypothesis being examined closely (index tc)
            int tc, chi;
            unsigned hi_excl;
            bool first = false;
            if (tau == 0x7f800000u) {
                // no best yet (the task's first hypothesis): its quartile, whatever it is
                const float vx = hyp[t], vy = hyp[32 + t], vz = hyp[64 + t];
                unsigned mx = 0u;
#pragma unroll
                for (int s = 0; s < SLOTS; ++s) {
                    const float r = fmaf(nz[s], vz, fmaf(ny[s], vy, nx[s] * vx));
                    sq[s] = r * r;
                    mx = max(mx, __float_as_uint(sq[s]));
                }
                mx = __reduce_max_sync(FULL, mx);
                if (mx >= 0x7f800000u) return kFastUndecided;
                hi_excl = mx + 1u;
                chi = NP;
                tc = t;
                first = true;
                t += 1;
            } else {
                const int t1 = (t + 1 < cnt) ? t + 1 : t;  // an odd batch ends with a doubled hypothesis
                const float2 vx2 = make_float2(hyp[t], hyp[t1]);
                const float2 vy2 = make_float2(hyp[32 + t], hyp[32 + t1]);
                const float2 vz2 = make_float2(hyp[64 + t], hyp[64 + t1]);
                const float2 nt2 = make_float2(nthr, nthr);
                float2 rr[SLOTS];
                unsigned c0 = 0, c1 = 0;
#pragma unroll
                for (int s = 0; s < SLOTS; ++s) {
                    float2 r = __fmul2_rn(vx2, make_float2(nx[s], nx[s]));
                    r = __ffma2_rn(vy2, make_float2(ny[s], ny[s]), r);
                    r = __ffma2_rn(vz2, make_float2(nz[s], nz[s]), r);
                    rr[s] = r;
                    const float2 e = __ffma2_rn(r, r, nt2);
                    c0 += __float_as_uint(e.x) >> 31;
                    c1 += __float_as_uint(e.y) >> 31;
                }
                const unsigned both = __reduce_add_sync(FULL, c0 | (c1 << 16));
                const int ca = (int)(both & 0xffffu), cb = (t1 != t) ? (int)(both >> 16) : 0;
                if (ca <= kk && cb <= kk) {  // both rigorously worse than the best so far
                    t += 2;
                    continue;
                }
                const bool second = ca <= kk;
                tc = second ? t1 : t;
                t += second ? 2 : 1;
                unsigned c = 0;
                const float nt = nthr;
#pragma unroll
                for (int s = 0; s < SLOTS; ++s) {
                    const float r = second ? rr[s].y : rr[s].x;
                    sq[s] = r * r;
                    c += __float_as_uint(sq[s] + nt) >> 31;
                }
                chi = (int)__reduce_add_sync(FULL, c);
                if (chi <= kk) continue;
                hi_excl = thr1;
            }
            const unsigned q = warp_select32<SLOTS>(sq, kk, hi_excl, chi, npad, n, first);
            const unsigned uq = up_bits(q);
            if (uq < tau) {  // rigorously better than the best so far
                tau = q;
                thr1 = uq + 1u;
                nthr = -__uint_as_float(thr1);
                has_real = true;
                M[0] = __shfl_sync(FULL, v[0], tc);
                M[1] = __shfl_sync(FULL, v[1], tc);
                M[2] = __shfl_sync(FULL, v[2], tc);
                continue;
            }
            if (!has_real) return kFastRetry;  // too close to a prior nobody holds: nothing to settle against
            // too close to the best so far to call in fp32 (cold): settle this one comparison with
            // the exact binary64 quartiles of the two hypotheses (a tie keeps the earlier one,
            // core_private.cpp:53), then resume
            const double tx = __shfl_sync(FULL, v[0], tc), ty = __shfl_sync(FULL, v[1], tc),
                         tz = __shfl_sync(FULL, v[2], tc);
            const unsigned long long qt = warp_exact_quartile<SLOTS>(w, n, lane, tx, ty, tz);
            const unsigned long long qb = warp_exact_quartile<SLOTS>(w, n, lane, M[0], M[1], M[2]);
            if (qt >= 0x7ff0000000000000ULL || qb >= 0x7ff0000000000000ULL) return kFastUndecided;
            if (settled) ++*settled;
            if (qt < qb) {
                tau = q;
                thr1 = uq + 1u;
                nthr = -__uint_as_float(thr1);
                M[0] = tx; M[1] = ty; M[2] = tz;
            }
        }
    }
    if (!has_real) return kFastRetry;  // nothing passed the prior
    if (tau_out) *tau_out = tau;
    return kFastOk;
}

// Phases B + C of an estimator task.  Returns kFlagP when the fp32 tournament could not take the rows (a
// row not finite, or too small to normalise): a hint only, the caller's cold path decides whether
// pre_sync's "non-finite numbers in P" condition holds (presync_diagnose).  prior / tau_out: see
// warp_ransac_fast (*tau_out = 0 when the winner did not come out of the fast path).
template <int SLOTS>
__device__ __forceinline__ unsigned warp_ransac(const DeviceData& dd, const FrameDesc& fd,
                                                const WarpSmem& w, int iters, uint64_t key, int lane,
                                                double M[3], unsigned* n_exact, unsigned prior = 0u,
                                                unsigned* tau_out = nullptr) {
    int settled = 0;
    FastStatus st = kFastRetry;
    unsigned tau = 0u;
    for (int attempt = 0; attempt < 2 && st == kFastRetry; ++attempt) {  // (one inlined copy of the tournament)
        st = warp_ransac_fast<SLOTS>(dd, fd, w, iters, key, lane, M, &settled, attempt == 0 ? prior : 0u, &tau);
        if (!prior) break;
    }
    if (tau_out) *tau_out = (st == kFastOk) ? tau : 0u;
    if (n_exact && settled && lane == 0) atomicAdd(n_exact, 1u);  // tasks that needed binary64
    if (st == kFastOk) return 0u;
    if (n_exact && !settled && lane == 0) atomicAdd(n_exact, 1u);
    const Vec3 e = warp_ransac_exact<SLOTS>(dd, fd, w, iters, key, lane);
    M[0] = e.x; M[1] = e.y; M[2] = e.z;
    return st == kFastRowsNotFinite ? kFlagP : 0u;
}

// ------------------------------------------------------------------------------------------
// FrameState::Loss 3-arg (core_private.cpp:117-123) on the warp's shared rows
__device__ __noinline__ double warp_loss3_smem(const double* __restrict__ sP, int NP, int nslots,
                                               int lane, double m0, double m1, double m2, double k,
                                               const double* __restrict__ tab) {
    const double scale = k / sqrt(dot3(m0, m1, m2, m0, m1, m2));
    double acc = 0.0;
    for (int s = 0; s < nslots; ++s) {
        const int i = s * 32 + lane;
        const double r = dot3(sP[i], sP[NP + i], sP[2 * NP + i], m0, m1, m2) * scale;
        acc = acc + log1p_nonneg(r * r, tab);  // padding rows are 0 -> log1p(0) = 0
    }
    return warp_sum(acc);
}

// Simplified (no-translation) loss mode, thesis pdf-p.27-28 section 2.11: the residual of a ray pair
// is |ar x br| itself -- the de-rotated rays of a purely rotating camera coincide -- instead of its
// component along the translation direction: sum_i log1p((|P_i| k)^2).  (The reference checkout has
// no code for it; the definition is this engine's and the oracle's, include/rssync_b200.h.)
__device__ __noinline__ double warp_loss_rows_smem(const double* __restrict__ sP, int NP, int nslots,
                                                   int lane, double k, const double* __restrict__ tab) {
    double acc = 0.0;
    for (int s = 0; s < nslots; ++s) {
        const int i = s * 32 + lane;
        const double p0 = sP[i], p1 = sP[NP + i], p2 = sP[2 * NP + i];
        const double r = sqrt(dot3(p0, p1, p2, p0, p1, p2)) * k;
        acc = acc + log1p_nonneg(r * r, tab);
    }
    return warp_sum(acc);
}
// arma::norm of the residual vector (the row norms)
__device__ __forceinline__ double warp_norm_rows(const double* sP, int NP, int nslots, int lane) {
    double ss = 0.0;
    for (int s = 0; s < nslots; ++s) {
        const int i = s * 32 + lane;
        const double p0 = sP[i], p1 = sP[NP + i], p2 = sP[2 * NP + i];
        const double nr = sqrt(dot3(p0, p1, p2, p0, p1, p2));
        ss = ss + nr * nr;
    }
    return sqrt(warp_sum(ss));
}

// FrameState::Loss 5-arg (core_private.cpp:92-115): value and d/dm in closed form of the
// forward-mode chain (inline_utils.hpp:19-48)
struct Loss5 {
    double f, g0, g1, g2;
};
__device__ __noinline__ Loss5 warp_loss5_smem(const double* __restrict__ sP, int NP, int nslots,
                                              int lane, double m0, double m1, double m2, double k,
                                              const double* __restrict__ tab) {
    const double kk = k * k;
    const double den = dot3(m0, m1, m2, m0, m1, m2) / kk;
    const double inv_den = 1.0 / den;
    double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};  // L, g0, g1, g2, su
    for (int s = 0; s < nslots; ++s) {
        const int i = s * 32 + lane;
        const double p0 = sP[i], p1 = sP[NP + i], p2 = sP[2 * NP + i];
        const double v1 = dot3(p0, p1, p2, m0, m1, m2);
        const double u = (v1 * v1) * inv_den;
        acc[0] = acc[0] + log1p_nonneg(u, tab);
        const double wgt = 1.0 / (1.0 + u);
        const double wv = wgt * v1;
        acc[1] = acc[1] + wv * p0;
        acc[2] = acc[2] + wv * p1;
        acc[3] = acc[3] + wv * p2;
        acc[4] = acc[4] + wgt * u;
    }
    warp_sum_n<5>(acc);
    Loss5 out;
    out.f = acc[0];
    const double G0 = acc[1], G1 = acc[2], G2 = acc[3];
    const double SU = acc[4];
    const double c1 = 2.0 * inv_den;
    const double c2 = (c1 / kk) * SU;
    out.g0 = c1 * G0 - c2 * m0;
    out.g1 = c1 * G1 - c2 * m1;
    out.g2 = c1 * G2 - c2 * m2;
    return out;
}

// Register-resident variants for the Sync kernels: the frame's rows stay in registers across all
// objective evaluations of one L-BFGS run (the delay, hence P, is fixed during it), the slot loops
// are compile-time so independent log1p / division chains interleave, and the five sums of an
// evaluation share one butterfly.  Same per-lane order of operations as the shared-memory variants
// above, hence the same bits (rows past the frame's end are zero and add exact zeros).
template <int SLOTS>
__device__ __forceinline__ void load_rows(const double* __restrict__ sP, int NP, int lane,
                                          double (&p)[SLOTS][3]) {
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
        const int i = s * 32 + lane;
        p[s][0] = sP[i];
        p[s][1] = sP[NP + i];
        p[s][2] = sP[2 * NP + i];
    }
}
template <int SLOTS>
__device__ __forceinline__ Loss5 warp_loss5_reg(const double (&p)[SLOTS][3], double m0, double m1,
                                                double m2, double k, const double* __restrict__ tab) {
    const double kk = k * k;
    const double den = dot3(m0, m1, m2, m0, m1, m2) / kk;
    const double inv_den = 1.0 / den;
    double v1[SLOTS], u[SLOTS], lg[SLOTS], wgt[SLOTS];
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
        v1[s] = dot3(p[s][0], p[s][1], p[s][2], m0, m1, m2);
        u[s] = (v1[s] * v1[s]) * inv_den;
    }
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
        lg[s] = log1p_nonneg(u[s], tab);
        wgt[s] = 1.0 / (1.0 + u[s]);
    }
    double r[5] = {0.0, 0.0, 0.0, 0.0, 0.0};  // L, g0, g1, g2, su
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
        const double wv = wgt[s] * v1[s];
        r[0] = r[0] + lg[s];
        r[1] = r[1] + wv * p[s][0];
        r[2] = r[2] + wv * p[s][1];
        r[3] = r[3] + wv * p[s][2];
        r[4] = r[4] + wgt[s] * u[s];
    }
    warp_sum_n<5>(r);
    Loss5 out;
    out.f = r[0];
    const double c1 = 2.0 * inv_den;
    const double c2 = (c1 / kk) * r[4];
    out.g0 = c1 * r[1] - c2 * m0;
    out.g1 = c1 * r[2] - c2 * m1;
    out.g2 = c1 * r[3] - c2 * m2;
    return out;
}
template <int SLOTS>
__device__ __forceinline__ double warp_loss3_reg(const double (&p)[SLOTS][3], double m0, double m1,
                                                 double m2, double k, const double* __restrict__ tab) {
    const double scale = k / sqrt(dot3(m0, m1, m2, m0, m1, m2));
    double lg[SLOTS];
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
        const double r = dot3(p[s][0], p[s][1], p[s][2], m0, m1, m2) * scale;
        lg[s] = log1p_nonneg(r * r, tab);
    }
    double acc = 0.0;
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) acc = acc + lg[s];
    return warp_sum(acc);
}

// ens::L_BFGS on a 3-vector (call site core_private.cpp:264-294); every lane runs the same scalar
// control flow on identical values, the objective is evaluated cooperatively.
// `hist`: kLbfgsHistDoubles doubles of shared memory private to the warp.  The stored pairs are
// indexed dynamically, so as local arrays they would live in local memory -- one copy per LANE of
// values that are identical in every lane (16 % of the kernel's stall samples were long-scoreboard
// waits on those loads).  Every lane writes every value itself before it reads it (all lanes write
// the same bits to the same address), so no warp synchronisation is needed.
constexpr int kLbfgsHistDoubles = 80;
template <class EvalF>
__device__ __forceinline__ double warp_lbfgs(EvalF&& eval, double x[3], int& n_iters, int& n_evals,
                                             double* __restrict__ hist) {
    constexpr int numBasis = 10, maxIterations = 200, maxTrials = 50;
    const double minGradientNorm = 1e-4, armijo = 1e-4, wolfe = 0.9, factr = 1e-15,
                 minStep = 1e-20, maxStep = 1e20;
    double (*S)[3] = reinterpret_cast<double (*)[3]>(hist);
    double (*Y)[3] = reinterpret_cast<double (*)[3]>(hist + 3 * numBasis);
    double* rho_pair = hist + 6 * numBasis;
    double* alpha = hist + 7 * numBasis;
    for (int i = 0; i < 7 * numBasis; ++i) hist[i] = 0.0;
    // 1 / (y.s) of each stored pair: the two-loop recursion recomputes this division for every pair
    // at every iteration; the value only depends on the pair, so it is computed once when the pair
    // is stored (same expression, same bits) -- it is the longest dependent chain of an iteration
    double g[3], oldx[3], oldg[3], dir[3], trial[3];
    Loss5 e = eval(x[0], x[1], x[2]);
    double f = e.f;
    g[0] = e.g0; g[1] = e.g1; g[2] = e.g2;
    n_evals = 1;
    n_iters = 0;
    for (int it = 0; it != maxIterations; ++it) {
        const double prevf = f;
        if (it > 0 && sqrt(dot3(g[0], g[1], g[2], g[0], g[1], g[2])) < minGradientNorm) break;
        if (f != f) break;
        // The two-loop recursion is a chain of dependent scalar FP64 operations (6 per stored pair
        // and loop); a frame that runs to maxIterations spends ~0.3 ms in it and its whole lane
        // waits.  The next pair is therefore loaded (shared memory, indices independent of the
        // chain) while the current one is being applied.
        const int cnt = (numBasis > it) ? it : numBasis;  // stored pairs in use
        int tp = (it + (numBasis - 1)) % numBasis;        // newest pair
        double s0 = S[tp][0], s1 = S[tp][1], s2 = S[tp][2];
        double y0 = Y[tp][0], y1 = Y[tp][1], y2 = Y[tp][2];
        double rp = rho_pair[tp];
        double scaling;
        if (it > 0) {
            const double yy = dot3(y0, y1, y2, y0, y1, y2);
            const double denom = (yy >= 1e-10) ? yy : 1.0;
            scaling = dot3(s0, s1, s2, y0, y1, y2) / denom;
        } else {
            const double gn = sqrt(dot3(g[0], g[1], g[2], g[0], g[1], g[2]));
            scaling = (gn >= 1e-5) ? 1.0 / gn : 1.0;
        }
        if (scaling == 0.0 || !is_finite(scaling)) break;
        dir[0] = g[0]; dir[1] = g[1]; dir[2] = g[2];
        for (int j = 0; j < cnt; ++j) {  // pairs it-1, it-2, ..., newest first
            const int tn = (tp == 0) ? numBasis - 1 : tp - 1;
            const double ns0 = S[tn][0], ns1 = S[tn][1], ns2 = S[tn][2];
            const double ny0 = Y[tn][0], ny1 = Y[tn][1], ny2 = Y[tn][2];
            const double nrp = rho_pair[tn];
            const double a = rp * dot3(s0, s1, s2, dir[0], dir[1], dir[2]);
            alpha[j] = a;
            dir[0] -= a * y0; dir[1] -= a * y1; dir[2] -= a * y2;
            s0 = ns0; s1 = ns1; s2 = ns2; y0 = ny0; y1 = ny1; y2 = ny2; rp = nrp;
            tp = tn;
        }
        for (int c = 0; c < 3; ++c) dir[c] *= scaling;
        tp = (it - cnt) % numBasis;  // oldest pair in use
        s0 = S[tp][0]; s1 = S[tp][1]; s2 = S[tp][2];
        y0 = Y[tp][0]; y1 = Y[tp][1]; y2 = Y[tp][2];
        rp = rho_pair[tp];
        for (int j = cnt - 1; j >= 0; --j) {  // oldest first
            const int tn = (tp == numBasis - 1) ? 0 : tp + 1;
            const double ns0 = S[tn][0], ns1 = S[tn][1], ns2 = S[tn][2];
            const double ny0 = Y[tn][0], ny1 = Y[tn][1], ny2 = Y[tn][2];
            const double nrp = rho_pair[tn];
            const double beta = rp * dot3(y0, y1, y2, dir[0], dir[1], dir[2]);
            const double coef = alpha[j] - beta;
            dir[0] += coef * s0; dir[1] += coef * s1; dir[2] += coef * s2;
            s0 = ns0; s1 = ns1; s2 = ns2; y0 = ny0; y1 = ny1; y2 = ny2; rp = nrp;
            tp = tn;
        }
        for (int c = 0; c < 3; ++c) dir[c] = -dir[c];
        for (int c = 0; c < 3; ++c) { oldx[c] = x[c]; oldg[c] = g[c]; }
        double step = 1.0, bestStep = 1.0, bestObj = 1.7976931348623157e308;
        const double init_dg = dot3(g[0], g[1], g[2], dir[0], dir[1], dir[2]);
        if (init_dg > 0.0) break;
        const double f0 = f;
        const double lin = armijo * init_dg;
        int trials = 0;
        for (;;) {
            for (int c = 0; c < 3; ++c) trial[c] = x[c] + step * dir[c];
            e = eval(trial[0], trial[1], trial[2]);
            f = e.f;
            g[0] = e.g0; g[1] = e.g1; g[2] = e.g2;
            n_evals++;
            if (f < bestObj) { bestStep = step; bestObj = f; }
            trials++;
            double width;
            if (f > f0 + step * lin) {
                width = 0.5;
            } else {
                const double dg = dot3(g[0], g[1], g[2], dir[0], dir[1], dir[2]);
                if (dg < wolfe * init_dg) width = 2.1;
                else if (dg > -wolfe * init_dg) width = 0.5;
                else break;
            }
            if (step < minStep || step > maxStep || trials >= maxTrials) break;
            step *= width;
        }
        for (int c = 0; c < 3; ++c) x[c] += bestStep * dir[c];
        n_iters++;
        if (bestStep == 0.0) break;
        const double denom = fmax(fmax(fabs(prevf), fabs(f)), 1.0);
        if ((prevf - f) / denom <= factr) break;
        const int op = it % numBasis;
        RS_ASSERT(op >= 0 && op < numBasis && cnt <= numBasis);
        for (int c = 0; c < 3; ++c) { S[op][c] = x[c] - oldx[c]; Y[op][c] = g[c] - oldg[c]; }
        const double ys = dot3(Y[op][0], Y[op][1], Y[op][2], S[op][0], S[op][1], S[op][2]);
        rho_pair[op] = (ys != 0) ? (1.0 / ys) : 1.0;
    }
    return f;
}

// arma::norm(P * M) over the warp (core_private.cpp:79,132); P.M goes to pm_out[i]
__device__ __forceinline__ double warp_norm_PM(const double* sP, int NP, int nslots, int lane,
                                               const double M[3], double* pm_out) {
    double ss = 0.0;
    for (int s = 0; s < nslots; ++s) {
        const int i = s * 32 + lane;
        const double pm = dot3(sP[i], sP[NP + i], sP[2 * NP + i], M[0], M[1], M[2]);
        if (pm_out) pm_out[i] = pm;
        ss = ss + pm * pm;
    }
    return sqrt(warp_sum(ss));
}

// which of pre_sync's panic conditions (core_private.cpp:76-83) a task hit; pm: the warp's rows, with
// P.M of each ray (simplified mode: the row's norm) in place of the first component (the loss phase
// leaves it there).  A non-finite row component makes P.M non-finite, and P.M of finite rows with the M
// the estimator draws from them (finite) is finite, so P.M and the other two planes tell whether a row
// is not finite (a row merely too small for the fp32 tournament is not)
__device__ __noinline__ unsigned presync_diagnose(const double* pm, int NP, int nslots, int lane, double scale,
                                                  double m0, double m1, double m2, const double* tab) {
    unsigned bad = 0;
    if (!(is_finite(m0) && is_finite(m1) && is_finite(m2))) bad |= kFlagM;
    for (int s = 0; s < nslots; ++s) {
        const int i = s * 32 + lane;
        if (!(is_finite(pm[i]) && is_finite(pm[NP + i]) && is_finite(pm[2 * NP + i]))) bad |= kFlagP;
        const double r = pm[i] * scale;
        if (!is_finite(r)) bad |= kFlagR;
        if (!is_finite(log1p_nonneg(r * r, tab))) bad |= kFlagRho;
    }
    return bad;
}

// ------------------------------------------------------------------------------------------
// K1: PreSync / DebugPreSync grid.
//
// Work unit = (frame, chunk of consecutive delays); a block walks a contiguous range of units, so
// consecutive units mostly share the frame.  What phase A reads is staged in shared memory by TMA bulk
// copies issued by one thread: the frame's ray tiles (contiguous in the arena) and the window of
// spline records the chunk can touch (from the frame's timestamp bounds and the chunk's delay
// range).  (With ~220 KB of the SM's 228 KB carved out as shared memory the L1 keeps a few KB:
// un-staged, the same loads hit L1 28 % of the time and wait on L2, profiles/r01_presync_v3c.md.)
//
// The staging area is a ring of two buffers and the block's warps take tasks from one shared
// counter, so nobody waits for anybody in the steady state:
//   * task k of the block is delay k % chunk of unit k / chunk; a warp that finishes a task takes
//     the next one (atomicAdd on next_task), whatever its neighbours are doing -- the lengths of the
//     estimator's tournaments differ from task to task, and with a static assignment (r01: warp j
//     takes delays j and j + W of a 16-delay unit, all warps meet at the unit's end) the block waited
//     for its slowest warp once per unit: 6 % of the warp samples on the staging mbarrier, 9 % of the
//     executed instructions in its polling loop (profiles/r01_presync_v6.md);
//   * unit u lives in buffer u & 1.  A buffer is live only during phase A of its unit's tasks: the
//     warp that completes the unit's last phase A (done_a counts them, whoever runs them) issues the
//     copies for unit u + 2 into it (`fence.proxy.async` first).  By then the data of unit u + 1 has
//     long landed -- it was requested a whole unit earlier -- so in the steady state a warp only
//     waits on the mbarrier during the block's first unit.  A warp entering unit u first waits until
//     the buffer has been handed to that unit (ctl->unit[b] == u: with short units a warp can be a
//     whole ring ahead of the buffer), then for the mbarrier phase of parity (u >> 1) & 1, which is
//     then unambiguous: the buffer is not handed on before all phase A's of unit u, that warp's
//     included.
// Grids with fewer delays per unit than the block has warps (a handful of delays over many frames)
// would serialise on the two buffers: they run unstaged (`staged` = 0), every task reading global
// memory through the general path, with no hand-off at all.
// A window that does not fit the buffer (delay steps of many samples, timestamps outside the gyro
// span) makes the unit read global memory through the out-of-line general path -- same arithmetic.
#ifndef RS_POLL_NS
#define RS_POLL_NS 64  // back-off between polls of a staging mbarrier
#endif
#ifndef RS_GRID_WARPS
#define RS_GRID_WARPS 8
#endif
#ifndef RS_GRID_MINB
#define RS_GRID_MINB 2
#endif
#ifndef RS_GRID_RECS
#define RS_GRID_RECS 128  // spline records per staged window (16 KB)
#endif
#ifndef RS_LOSS_UNROLL
#define RS_LOSS_UNROLL 4  // slots per iteration of the loss phase
#endif
#ifndef RS_GRID_GRAB
#define RS_GRID_GRAB 4    // consecutive tasks a warp takes from the block's counter at a time
#endif
#ifndef RS_GRID_PRIOR
#define RS_GRID_PRIOR 1   // start each tournament from the neighbouring delay's winning quartile
#endif
#ifndef RS_PRIOR_BUMP
#define RS_PRIOR_BUMP 0x00800000u  // added to the prior's bit pattern: one exponent = x 2
#endif
template <int SLOTS>
struct GridCfg {
    static constexpr int kWarps = RS_GRID_WARPS;
    static constexpr int kMinBlocks = SLOTS <= 8 ? RS_GRID_MINB : 1;
    static constexpr size_t kTileBytes = (size_t)SLOTS * 2048;
    // spline records per staged window: what kMinBlocks blocks leave of the SM's 228 KB (1 KB per
    // block is the system's), in steps of 8 records, at most RS_GRID_RECS
    static constexpr long long kRoom = (228 * 1024) / kMinBlocks - 1024 - (long long)kLog1pTableBytes - 256 -
                                       (long long)kWarps * (long long)warp_smem_bytes(SLOTS * 32) - 2 * (long long)kTileBytes;
    static constexpr int kRecsFit = (int)(kRoom / 256 / 8 * 8);
    static constexpr int kRecs = kRecsFit < RS_GRID_RECS ? kRecsFit : RS_GRID_RECS;
    static_assert(kRecs >= 40, "grid kernel: no room for a spline window");
    static constexpr size_t kBufBytes = kTileBytes + (size_t)kRecs * 128;
    static constexpr size_t kCtlOff = kLog1pTableBytes;
    static constexpr size_t kBufOff = kCtlOff + 256;
    static constexpr size_t kWarpOff = kBufOff + 2 * kBufBytes;
    static constexpr size_t kSmem = kWarpOff + (size_t)kWarps * warp_smem_bytes(SLOTS * 32);
    // kMinBlocks blocks must fit the SM's 228 KB (1 KB per block is the system's)
    static_assert(kMinBlocks * (kSmem + 1024) <= 228 * 1024, "grid kernel: shared memory over budget");
};
struct GridCtl {
    unsigned long long full[2];  // mbarriers: the staged data of the unit in buffer b has landed
    int done_a[2];               // phase A's completed in the unit occupying buffer b
    int next_task;               // the block's task counter
    int rec_first[2], rec_cnt[2];  // staged spline window; rec_cnt = 0: not staged, phase A reads global
    int frame[2], d0[2];         // the unit's frame (index into `frames`) and first delay
    int unit[2];                 // which unit of the block buffer b belongs to (-1: none yet)
    FrameDesc fd[2];
};
static_assert(sizeof(GridCtl) <= 256, "GridCtl must fit its slot");

// issue the copies of unit (fi, ci) into buffer b; one thread
__device__ __noinline__ void grid_stage_unit(const DeviceData& dd, const FrameDesc* frames,
                                             const double* delays, int D, int chunk, int fi, int ci, int u,
                                             GridCtl* ctl, int b, double* sTiles, double* sRec, int rec_cap) {
    const int d0 = ci * chunk;
    const int d1 = min(D, d0 + chunk);
    const FrameDesc fd = frames[fi];
    double dmin = delays[d0], dmax = dmin;
    for (int d = d0 + 1; d < d1; ++d) {
        dmin = fmin(dmin, delays[d]);
        dmax = fmax(dmax, delays[d]);
    }
    // x = ((ts - q0) + delay) * sr is monotone in ts and in delay, roundings included
    const double x_lo = ((fd.ts_lo - dd.q0) + dmin) * dd.sr, x_hi = ((fd.ts_hi - dd.q0) + dmax) * dd.sr;
    const double r_lo = floor(x_lo) - 1.0, r_hi = floor(x_hi) + 2.0;  // a record of slack either side
    const bool ok = dd.sr > 0.0 && r_lo >= 0.0 && r_hi <= (double)(dd.nq - 1) && (r_hi - r_lo) < (double)rec_cap;
    const int first = ok ? (int)r_lo : 0, cnt = ok ? (int)(r_hi - r_lo) + 1 : 0;
    ctl->rec_first[b] = first;
    ctl->rec_cnt[b] = cnt;
    ctl->frame[b] = fi;
    ctl->d0[b] = d0;
    ctl->fd[b] = fd;
    __threadfence_block();
    *(volatile int*)&ctl->unit[b] = u;  // after the unit's parameters: a waiter reads them once it sees u
    // the buffer was read through the generic proxy; order those reads before the async writes
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    const unsigned tile_bytes = (unsigned)((fd.n + 31) >> 5) * 2048u;
    const unsigned bytes = ok ? (unsigned)cnt * 128u + tile_bytes : 0u;
    mbar_arrive_expect_tx(&ctl->full[b], bytes);
    if (ok) {
        tma_load_1d(sRec, dd.rec + (size_t)first * 16, (unsigned)cnt * 128u, &ctl->full[b]);
        tma_load_1d(sTiles, dd.rays + (size_t)fd.off * 8, tile_bytes, &ctl->full[b]);
    }
}

// SIMPLE: the simplified (no-translation) loss mode, a separate instantiation so that the
// reference's path carries none of its branches
template <int SLOTS, bool SIMPLE>
__global__ void __launch_bounds__(GridCfg<SLOTS>::kWarps * 32, GridCfg<SLOTS>::kMinBlocks)
presync_kernel(DeviceData dd, const FrameDesc* __restrict__ frames, int F,
               const double* __restrict__ delays, int D, int chunk, int cpf, uint64_t seed,
               uint64_t stream, uint64_t call_no, const uint64_t* __restrict__ frame_call_no,
               uint64_t idx_base, double* __restrict__ framecost, int cost_stride,
               unsigned* __restrict__ flags, int staged) {
    using Cfg = GridCfg<SLOTS>;
    constexpr bool simplified = SIMPLE;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int NP = SLOTS * 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* tab = reinterpret_cast<double*>(smem_raw);
    GridCtl* ctl = reinterpret_cast<GridCtl*>(smem_raw + Cfg::kCtlOff);
    unsigned char* bufs = smem_raw + Cfg::kBufOff;
    const WarpSmem w = warp_smem(smem_raw + Cfg::kWarpOff, warp, NP);
    // units are counted in 64 bits (the host accepts grids up to 2^40 tasks); a block's share fits an int
    const long long U = (long long)F * cpf;
    const long long u_begin = U * blockIdx.x / gridDim.x;
    const int n_units = (int)(U * (blockIdx.x + 1) / gridDim.x - u_begin);
    const int fi0 = (int)(u_begin / cpf), c0 = (int)(u_begin % cpf);
    auto stage = [&](int u) {
        const int cu = c0 + u, b = u & 1;
        double* sTiles = reinterpret_cast<double*>(bufs + (size_t)b * Cfg::kBufBytes);
        grid_stage_unit(dd, frames, delays, D, chunk, fi0 + cu / cpf, cu % cpf, u, ctl, b, sTiles,
                        sTiles + SLOTS * 256, Cfg::kRecs);
    };
    if (threadIdx.x == 0) {
        mbar_init(&ctl->full[0], 1);
        mbar_init(&ctl->full[1], 1);
        ctl->done_a[0] = ctl->done_a[1] = 0;
        ctl->unit[0] = ctl->unit[1] = -1;
        ctl->next_task = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    load_log1p_table(tab);  // ends with __syncthreads()
    if (threadIdx.x == 0 && staged) {
        if (n_units > 0) stage(0);
        if (n_units > 1) stage(1);
    }
    const int n_tasks = n_units * chunk;  // the host keeps a grid below 2^34 tasks
    int cur_u = -1, rec_first = 0, rec_cnt = 0, fi = 0, d0 = 0;
    FrameDesc fd{};
    // A warp takes kGrab consecutive tasks at a time: consecutive delays of one frame, so that the
    // estimator of each can start from its predecessor's winning quartile (warp_ransac_fast, `prior`).
    unsigned prior = 0u;
    int prior_u = -1, prior_dj = -2;
    for (int k_next = 0, k_end = 0;;) {
        if (k_next == k_end) {
            if (lane == 0) k_next = atomicAdd(&ctl->next_task, RS_GRID_GRAB);
            k_next = __shfl_sync(FULL, k_next, 0);
            k_end = min(k_next + RS_GRID_GRAB, n_tasks);
            if (k_next >= n_tasks) break;
        }
        const int k = k_next++;
        const int u = k / chunk, dj = k - u * chunk;
        const int b = u & 1;
        if (u != cur_u && !staged) {
            cur_u = u;
            const int cu = c0 + u;
            fi = fi0 + cu / cpf;
            d0 = (cu % cpf) * chunk;
            fd = frames[fi];
        } else if (u != cur_u) {  // first task this warp takes in unit u
            cur_u = u;
#ifdef RS_CHECKED
            unsigned spins = 0;
#endif
            for (int have; (have = *(volatile int*)&ctl->unit[b]) != u;) {
                RS_ASSERT(++spins < (1u << 24) && have < u);  // never handed past a unit still needed
                __nanosleep(RS_POLL_NS);
            }
            const unsigned parity = (unsigned)(u >> 1) & 1u;
            while (!mbar_try_wait(&ctl->full[b], parity)) {
                RS_ASSERT(++spins < (1u << 24));
                __nanosleep(RS_POLL_NS);
            }
            RS_ASSERT(*(volatile int*)&ctl->unit[b] == u);
            rec_first = *(volatile int*)&ctl->rec_first[b];
            rec_cnt = *(volatile int*)&ctl->rec_cnt[b];
            fi = *(volatile int*)&ctl->frame[b];
            d0 = *(volatile int*)&ctl->d0[b];
            const volatile FrameDesc* vf = &ctl->fd[b];
            fd.id = vf->id; fd.off = vf->off; fd.n = vf->n; fd.ts_lo = vf->ts_lo; fd.ts_hi = vf->ts_hi;
        }
        const int di = d0 + dj;
        const bool active = di < D;
        RS_ASSERT(fi >= 0 && fi < F && dj >= 0 && dj < chunk && fd.n >= 2 && fd.n <= NP);
        double delay = 0.0;
        if (active) {
            delay = delays[di];
            const double* sTiles = reinterpret_cast<const double*>(bufs + (size_t)b * Cfg::kBufBytes);
            if (rec_cnt) build_rows_staged(dd, fd, delay, lane, w, NP, sTiles, sTiles + SLOTS * 256, rec_first, rec_cnt);
            else build_rows_global_cold(dd, fd, delay, lane, w, NP);
        }
        __syncwarp();
        if (lane == 0 && staged) {  // this phase A no longer needs the staging buffer
            __threadfence_block();
            RS_ASSERT(*(volatile int*)&ctl->unit[b] == u);  // the buffer was not handed on under this phase A
            const int done = atomicAdd(&ctl->done_a[b], 1);
            RS_ASSERT(done >= 0 && done < chunk);
            if (done == chunk - 1) {  // the unit's last: refill the buffer
                ctl->done_a[b] = 0;
                if (u + 2 < n_units) stage(u + 2);
            }
        }
        if (!active) continue;
        const uint64_t key =
            rng_task_key(rng_prefix(seed, stream, frame_call_no ? frame_call_no[fi] : call_no,
                                    idx_base + (uint64_t)di),
                         fd.id);
        double M[3] = {0.0, 0.0, 0.0};
        unsigned bad = 0u;
        if (!simplified) {
            // prior: twice the neighbouring delay's winning quartile (one more exponent; the winning
            // quartile moves by less than 2 x between neighbouring delays 98.75 % of the time)
            const bool neighbour = RS_GRID_PRIOR && prior && prior_u == u && prior_dj + 1 == dj && prior < 0x7e000000u;
            unsigned tau = 0u;
            bad = warp_ransac<SLOTS>(dd, fd, w, 20, key, lane, M, flags + 1, neighbour ? prior + RS_PRIOR_BUMP : 0u,
                                     &tau);  // core_private.cpp:77
            prior = tau;
            prior_u = u;
            prior_dj = dj;
        }
        // :79-85
        __syncwarp();
        // rows past the frame's last ray are zero: they add 0 to the norm and log1p(0) = 0 to the loss.
        // Written as loops over groups of kLossUnroll slots (independent chains inside a group):
        // the fully unrolled form is 7 KB of straight-line code that every task streams through the
        // instruction caches once.  P.M of a ray replaces the ray's first row component in shared
        // memory between the two passes (each lane touches only its own rays).
        constexpr int LU = RS_LOSS_UNROLL < SLOTS ? RS_LOSS_UNROLL : SLOTS;
        double ss = 0.0;
#pragma unroll 1
        for (int s0 = 0; s0 < SLOTS; s0 += LU) {
            double pm[LU];
#pragma unroll
            for (int j = 0; j < LU; ++j) {
                const int i = (s0 + j) * 32 + lane;
                pm[j] = 0.0;
                if (s0 + j < SLOTS) {
                    const double p0 = w.P[i], p1 = w.P[NP + i], p2 = w.P[2 * NP + i];
                    // simplified mode: the residual is the row's norm
                    pm[j] = simplified ? sqrt(dot3(p0, p1, p2, p0, p1, p2)) : dot3(p0, p1, p2, M[0], M[1], M[2]);
                    w.P[i] = pm[j];
                }
            }
#pragma unroll
            for (int j = 0; j < LU; ++j) ss = ss + pm[j] * pm[j];
        }
        const double kv = clamp_k(1.0 / sqrt(warp_sum(ss)) * 1e2);  // arma::norm(P * M), :79
        const double scale = simplified ? kv : kv / sqrt(dot3(M[0], M[1], M[2], M[0], M[1], M[2]));
        double acc = 0.0;
#pragma unroll 1
        for (int s0 = 0; s0 < SLOTS; s0 += LU) {
            double rho[LU];
#pragma unroll
            for (int j = 0; j < LU; ++j) {
                const double r = (s0 + j < SLOTS ? w.P[(s0 + j) * 32 + lane] : 0.0) * scale;
                rho[j] = sqrt(log1p_nonneg(r * r, tab));
            }
#pragma unroll
            for (int j = 0; j < LU; ++j) acc = acc + rho[j];
        }
        const double cost = sqrt(warp_sum(acc));
        if (lane == 0) framecost[(size_t)di * cost_stride + fi] = cost;
        // the panic conditions of :76-83: non-finite values propagate into the cost, so the stage
        // that produced them is only looked for when the cost is not finite or the estimator could not
        // take the rows (bad: non-finite rows, or rows too small for fp32, which are no panic)
        if (bad || !is_finite(cost)) {
            bad = presync_diagnose(w.P, NP, (fd.n + 31) >> 5, lane, scale, M[0], M[1], M[2], tab);
            bad = __reduce_or_sync(FULL, bad);
            if (bad && lane == 0) atomicOr(flags, bad);
        }
    }
}

// cost[d] = double-double sum over frames of framecost[d][.]  (the mutex-guarded `cost +=` of
// core_private.cpp:84-85); one warp per delay.
__global__ void reduce_rows_kernel(const double* __restrict__ in, int rows, int cols,
                                   double* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    DD acc = dd_zero();
    for (int c = lane; c < cols; c += 32) dd_add(acc, in[(size_t)row * cols + c]);
    const double v = warp_dd_sum(acc);
    if (lane == 0) out[row] = v;
}

// several PreSync windows in one grid: cost[w][d] = double-double sum of framecost[d][f] over the
// window's frames f in [win_begin[w], win_begin[w + 1]); one warp per (window, delay)
__global__ void reduce_windows_kernel(const double* __restrict__ in, int D, int F,
                                      const int* __restrict__ win_begin, int W,
                                      double* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= W * D) return;
    const int wi = q / D, d = q % D;
    DD acc = dd_zero();
    for (int f = win_begin[wi] + lane; f < win_begin[wi + 1]; f += 32) dd_add(acc, in[(size_t)d * F + f]);
    const double v = warp_dd_sum(acc);
    if (lane == 0) out[q] = v;
}

// ------------------------------------------------------------------------------------------
// K4: Sync initialisation, GuessMotion (RANSAC-200) + GuessK per (syncpoint, frame) task
template <int SLOTS>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
sync_init_kernel(DeviceData dd, SyncBatchDev b, const double* __restrict__ sp_delay,
                 const uint64_t* __restrict__ sp_callno, const unsigned char* __restrict__ sp_active,
                 uint64_t seed) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int NP = SLOTS * 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const WarpSmem w = warp_smem(smem_raw, warp, NP);
    for (int t = blockIdx.x * kWarpsPerBlock + warp; t < b.T; t += gridDim.x * kWarpsPerBlock) {
        const SyncTask task = b.tasks[t];
        if (!sp_active[task.sp]) continue;
        const int nslots = (task.fd.n + 31) >> 5;
        __syncwarp();
        build_rows_smem(dd, task.fd, sp_delay[task.sp], lane, w, NP);
        if (b.simplified) {  // no translation direction: only the scale, from the row norms
            const double nr = warp_norm_rows(w.P, NP, nslots, lane);
            if (lane == 0) {
                b.m[3 * t + 0] = 0.0; b.m[3 * t + 1] = 0.0; b.m[3 * t + 2] = 0.0;
                b.k[t] = clamp_k(1.0 / nr * 1e2);
            }
            continue;
        }
        const uint64_t key =
            rng_task_key(rng_prefix(seed, kStreamSyncInit, sp_callno[task.sp], 0), task.fd.id);
        double M[3];
        warp_ransac<SLOTS>(dd, task.fd, w, 200, key, lane, M, nullptr);  // core_private.cpp:127
        __syncwarp();
        const double nrm = warp_norm_PM(w.P, NP, nslots, lane, M, nullptr);
        if (lane == 0) {
            b.m[3 * t + 0] = M[0]; b.m[3 * t + 1] = M[1]; b.m[3 * t + 2] = M[2];
            b.k[t] = clamp_k(1.0 / nrm * 1e2);  // :132
        }
    }
}

// K2+K3a: per task, L-BFGS refinement of m at the syncpoint's delay (do_opt_motion, :262-296), then
// the three objective values the delay step needs (Loss5 at x0, Loss3 at x0 -/+ h, :228-240).
#ifndef RS_SYNC_MINB
#define RS_SYNC_MINB 1
#endif
// Two builds.  The kernel needs ~200 registers per thread (the frame's rows stay in registers across
// the L-BFGS evaluations): eight-warp blocks, one per SM, uncapped -- the fastest for a straggler,
// which is what bounds a small batch (C2: 27 syncpoints); and two-warp blocks capped at 168
// registers, twelve warps per SM -- each warp ~8 % slower, but half as many waves when the batch
// has many more frame tasks than the device has warp slots (C4).  The host picks by task count.
template <bool SMALL>
struct LbfgsCfg {
    static constexpr int kWarps = SMALL ? 2 : kWarpsPerBlock;
    static constexpr int kMinBlocks = SMALL ? 6 : RS_SYNC_MINB;
};
template <int SLOTS, bool SMALL>
__global__ void __launch_bounds__(LbfgsCfg<SMALL>::kWarps * 32, SLOTS <= 8 ? LbfgsCfg<SMALL>::kMinBlocks : 1)
sync_motion_fgrad_kernel(DeviceData dd, SyncBatchDev b, const double* __restrict__ sp_delay,
                         const double* __restrict__ sp_x0,
                         const unsigned char* __restrict__ sp_active, double* __restrict__ scratch,
                         int* __restrict__ stats, unsigned long long* __restrict__ evals_total) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int NP = SLOTS * 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* tab = reinterpret_cast<double*>(smem_raw);
    load_log1p_table(tab);
    const WarpSmem w = warp_smem(smem_raw + kLog1pTableBytes, warp, NP);
    constexpr int W = LbfgsCfg<SMALL>::kWarps;
    double* hist = reinterpret_cast<double*>(smem_raw + kLog1pTableBytes + (size_t)W * warp_smem_bytes(NP)) +
                   warp * kLbfgsHistDoubles;
    for (int t = blockIdx.x * W + warp; t < b.T; t += gridDim.x * W) {
        const SyncTask task = b.tasks[t];
        if (!sp_active[task.sp]) continue;
        double m[3] = {b.m[3 * t], b.m[3 * t + 1], b.m[3 * t + 2]};
        const double k = b.k[t];
        const double x0 = sp_x0[task.sp];
        for (int j = b.simplified ? 1 : 0; j < 4; ++j) {  // (simplified mode: no direction to refine)
            const double delay = (j == 0)   ? sp_delay[task.sp]
                                 : (j == 1) ? x0
                                 : (j == 2) ? x0 - kNumericDiffStep
                                            : x0 + kNumericDiffStep;
            __syncwarp();
            build_rows_smem(dd, task.fd, delay, lane, w, NP);
            double p[SLOTS][3];
            load_rows<SLOTS>(w.P, NP, lane, p);
            if (j == 0) {
                int it, ev;
                warp_lbfgs([&](double a0, double a1, double a2) { return warp_loss5_reg<SLOTS>(p, a0, a1, a2, k, tab); },
                           m, it, ev, hist);
                if (lane == 0) {
                    b.m[3 * t] = m[0]; b.m[3 * t + 1] = m[1]; b.m[3 * t + 2] = m[2];
                    if (stats) { stats[2 * t] = it; stats[2 * t + 1] = ev; }
                    if (evals_total) atomicAdd(evals_total, (unsigned long long)ev);
                }
            } else if (b.simplified) {
                const double v = warp_loss_rows_smem(w.P, NP, (task.fd.n + 31) >> 5, lane, k, tab);
                if (lane == 0) scratch[3 * t + (j - 1)] = v;
            } else if (j == 1) {
                const Loss5 e = warp_loss5_reg<SLOTS>(p, m[0], m[1], m[2], k, tab);
                if (lane == 0) scratch[3 * t] = e.f;
            } else {
                const double v = warp_loss3_reg<SLOTS>(p, m[0], m[1], m[2], k, tab);
                if (lane == 0) scratch[3 * t + (j - 1)] = v;
            }
        }
    }
}

// sum over the frame's rays of NVAL per-ray terms held one ray per thread (block of SLOTS warps), in
// the contract's order: lane partial sums over the slots from 0.0, then the xor butterfly
// per syncpoint: cost = sum v, grad = sum (r - l)/2/h   (core_private.cpp:112, 236-237)
// and the trial points of Backtrack::Step (backtrack.cpp:5-12: t = initial_step, then t *= decay),
// x0 - t g with the hyper-parameters of core_private.cpp:226: every trial point is known once the
// gradient is, so the trial kernel follows in the stream without a host round trip
__global__ void reduce_fgrad_kernel(SyncBatchDev b, const unsigned char* __restrict__ sp_active,
                                    const double* __restrict__ scratch, const double* __restrict__ sp_x0,
                                    double* __restrict__ out_v, double* __restrict__ out_g,
                                    double* __restrict__ trial_delay, int ntrial) {
    const int lane = threadIdx.x & 31;
    const int sp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (sp >= b.S || !sp_active[sp]) return;
    DD av = dd_zero(), ag = dd_zero();
    for (int t = b.sp_begin[sp] + lane; t < b.sp_begin[sp + 1]; t += 32) {
        dd_add(av, scratch[3 * t]);
        dd_add(ag, (scratch[3 * t + 2] - scratch[3 * t + 1]) / 2 / kNumericDiffStep);
    }
    const double v = warp_dd_sum(av), g = warp_dd_sum(ag);
    if (lane == 0) {
        out_v[sp] = v;
        out_g[sp] = g;
        const double x0 = sp_x0[sp];
        double t = 1e-3;
        for (int i = 0; i < ntrial; ++i) {
            trial_delay[(size_t)sp * ntrial + i] = x0 - t * g;
            t *= .1;
        }
    }
}

// K3b: Loss3 at ntrial delays per syncpoint (backtracking trial points / final objective)
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
sync_trials_kernel(DeviceData dd, SyncBatchDev b, int NP, const double* __restrict__ trial_delay,
                   int ntrial, const unsigned char* __restrict__ sp_active,
                   double* __restrict__ scratch, const double* __restrict__ n_eval) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* tab = reinterpret_cast<double*>(smem_raw);
    load_log1p_table(tab);
    const WarpSmem w = warp_smem(smem_raw + kLog1pTableBytes, warp, NP);
    const long long total = (long long)b.T * ntrial;
    for (long long q = (long long)blockIdx.x * kWarpsPerBlock + warp; q < total;
         q += (long long)gridDim.x * kWarpsPerBlock) {
        const int t = (int)(q / ntrial), j = (int)(q % ntrial);
        // only the first *n_eval trial points are evaluated (the host's guess of how far Backtrack
        // will get; it asks for the rest when the guess was short)
        if (n_eval && j >= (int)*n_eval) continue;
        const SyncTask task = b.tasks[t];
        if (!sp_active[task.sp]) continue;
        const int nslots = (task.fd.n + 31) >> 5;
        __syncwarp();
        build_rows_smem(dd, task.fd, trial_delay[(size_t)task.sp * ntrial + j], lane, w, NP);
        const double v = b.simplified ? warp_loss_rows_smem(w.P, NP, nslots, lane, b.k[t], tab)
                                      : warp_loss3_smem(w.P, NP, nslots, lane, b.m[3 * t], b.m[3 * t + 1],
                                                        b.m[3 * t + 2], b.k[t], tab);
        if (lane == 0) scratch[(size_t)t * ntrial + j] = v;
    }
}

__global__ void reduce_trials_kernel(SyncBatchDev b, int ntrial,
                                     const unsigned char* __restrict__ sp_active,
                                     const double* __restrict__ scratch, double* __restrict__ out,
                                     const double* __restrict__ n_eval) {
    const int lane = threadIdx.x & 31;
    const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= b.S * ntrial) return;
    const int sp = q / ntrial, j = q % ntrial;
    if (!sp_active[sp] || (n_eval && j >= (int)*n_eval)) return;
    DD acc = dd_zero();
    for (int t = b.sp_begin[sp] + lane; t < b.sp_begin[sp + 1]; t += 32)
        dd_add(acc, scratch[(size_t)t * ntrial + j]);
    const double v = warp_dd_sum(acc);
    if (lane == 0) out[(size_t)sp * ntrial + j] = v;
}

// ------------------------------------------------------------------------------------------
// K6: pixel -> ray front end.  lens_undistort_point (core_testcode.cpp:63-95): fisheye model
// theta_d = theta (1 + k1 theta^2 + ...), inverted by 9 Newton steps from pi/4 -- including the
// reference's derivative coefficient 8 k4 (:80; 9 k4 would be the exact one, it only changes the
// convergence speed) and its halving loop that keeps theta inside (0, pi/2).
__device__ __forceinline__ void undistort_point(const LensDev& L, double px, double py, double& ux,
                                                double& uy) {
    if (sqrt(px * px + py * py) < 1e-8) { ux = 0.0; uy = 0.0; return; }  // :64
    const double x_ = (px - L.cx) / L.fx, y_ = (py - L.cy) / L.fy;
    const double theta_ = sqrt(x_ * x_ + y_ * y_);
    const double kPi = 3.14159265358979323846;
    double theta = kPi / 4.;
    for (int i = 0; i < 9; ++i) {
        const double t2 = theta * theta, t3 = t2 * theta, t4 = t2 * t2, t5 = t2 * t3, t6 = t3 * t3,
                     t7 = t3 * t4, t8 = t4 * t4, t9 = t4 * t5;
        const double cur = theta + L.k1 * t3 + L.k2 * t5 + L.k3 * t7 + L.k4 * t9;
        const double dcur = 1 + 3 * L.k1 * t2 + 5 * L.k2 * t4 + 7 * L.k3 * t6 + 8 * L.k4 * t8;
        const double err = cur - theta_;
        double nt = theta - err * (1. / dcur);
        for (int guard = 0; (nt >= kPi / 2. || nt <= 0.) && guard < 2048; ++guard) nt = (nt + theta) / 2.;
        theta = nt;
    }
    const double r = tan(theta), inv_cos = 1. / cos(theta);
    const double s = (theta_ < 1e-9) ? inv_cos : r / theta_;
    ux = x_ * s;
    uy = y_ * s;
}

constexpr int kIngestThreads = 256;
// block-wide: sort the frame's points by (ts_a, caller index) -- the order std::sort gives the host
// path -- and write the frame's tiles [8 fields][32 rays] and its orig / pos planes to the arena
__device__ __forceinline__ void ingest_sort_and_store(const PixelFrame& f, const double* s_ts, int* s_idx,
                                                      const double (*s_val)[kMaxRaysPerFrame],
                                                      double* __restrict__ rays, int32_t* __restrict__ orig,
                                                      int32_t* __restrict__ pos) {
    int nsort = 32;  // power of two covering the frame
    while (nsort < f.n) nsort <<= 1;
    for (int k = 2; k <= nsort; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < nsort; i += kIngestThreads) {
                const int l = i ^ j;
                if (l > i) {
                    const int a = s_idx[i], b = s_idx[l];
                    const double ta = s_ts[a], tb = s_ts[b];
                    const bool a_first = ta < tb || (ta == tb && a < b);
                    const bool up = (i & k) == 0;
                    if (a_first != up) { s_idx[i] = b; s_idx[l] = a; }
                }
            }
            __syncthreads();
        }
    const int padded = (f.n + 31) / 32 * 32;
    for (int j = threadIdx.x; j < padded; j += kIngestThreads) {
        double* t = rays + ((size_t)f.off + (j & ~31)) * 8 + (j & 31);
        if (j < f.n) {
            const int i = s_idx[j];
            orig[f.off + j] = i;
            pos[f.off + i] = j;
            t[0] = s_ts[i];
#pragma unroll
            for (int c = 0; c < 7; ++c) t[32 * (c + 1)] = s_val[c][i];
        } else {  // padding lanes: finite, masked out by n (same fill as the host path)
            const int last = f.n ? s_idx[f.n - 1] : 0;
            orig[f.off + j] = j;
            pos[f.off + j] = j;
            t[0] = f.n ? s_ts[last] : 0.0;
            t[32] = f.n ? s_val[0][last] : 0.0;
#pragma unroll
            for (int c = 2; c < 8; ++c) t[32 * c] = 0.0;
        }
    }
}
__global__ void __launch_bounds__(kIngestThreads)
ingest_pixels_kernel(const PixelFrame* __restrict__ frames, const double* __restrict__ pa,
                     const double* __restrict__ pb, LensDev L, double rows, double* __restrict__ rays,
                     int32_t* __restrict__ orig, int32_t* __restrict__ pos, double2* __restrict__ rowq) {
    __shared__ double s_ts[kMaxRaysPerFrame];  // ts_a of point i (sort key)
    __shared__ int s_idx[kMaxRaysPerFrame];    // permutation being sorted
    __shared__ double s_val[7][kMaxRaysPerFrame];  // ts_b, ra.xyz, rb.xyz of point i
    const PixelFrame f = frames[blockIdx.x];
    for (int i = threadIdx.x; i < kMaxRaysPerFrame; i += kIngestThreads) {
        s_idx[i] = i;
        if (i < f.n) {
            const double ax = pa[2 * (f.src + i)], ay = pa[2 * (f.src + i) + 1];
            const double bx = pb[2 * (f.src + i)], by = pb[2 * (f.src + i) + 1];
            double ua, va, ub, vb;
            undistort_point(L, ax, ay, ua, va);
            undistort_point(L, bx, by, ub, vb);
            const double qa = ay / rows, qb = by / rows;
            rowq[f.off + i] = make_double2(qa, qb);  // kept for re-timing (retime_frames_kernel)
            s_ts[i] = f.ts_a + L.ro * qa;  // :144
            s_val[0][i] = f.ts_b + L.ro * qb;  // :145
            const double na = sqrt(ua * ua + va * va + 1.0), nb = sqrt(ub * ub + vb * vb + 1.0);
            s_val[1][i] = ua / na; s_val[2][i] = va / na; s_val[3][i] = 1.0 / na;  // :153
            s_val[4][i] = ub / nb; s_val[5][i] = vb / nb; s_val[6][i] = 1.0 / nb;  // :154
        } else {
            s_ts[i] = __longlong_as_double(0x7ff0000000000000LL);  // padding sorts last
        }
    }
    __syncthreads();
    ingest_sort_and_store(f, s_ts, s_idx, s_val, rays, orig, pos);
}

// Rolling-shutter re-timing of frames ingested from pixels: the rays stay, the timestamps are
// recomputed at readout `ro` from the row fractions ingest_pixels_kernel kept (rowq[off + i] = {y_a,
// y_b} / rows of caller ray i), with its expression, and the frame is sorted and stored again.
// f.src: the frame's offset in the source arena, f.off: in the destination arena (the same arena is
// allowed: the block holds the whole frame in shared memory before it writes).  ext (optional): per
// frame the smallest / largest q_a and q_b, from which the host derives the frame's timestamp bounds.
__global__ void __launch_bounds__(kIngestThreads)
retime_frames_kernel(const PixelFrame* __restrict__ frames, const double* src_rays, const int32_t* src_orig,
                     const double2* __restrict__ rowq, double ro, double* rays, int32_t* orig, int32_t* pos,
                     double4* __restrict__ ext) {
    __shared__ double s_ts[kMaxRaysPerFrame];
    __shared__ int s_idx[kMaxRaysPerFrame];
    __shared__ double s_val[7][kMaxRaysPerFrame];
    __shared__ double s_ext[kIngestThreads / 32][4];
    const PixelFrame f = frames[blockIdx.x];
    RS_ASSERT(f.n >= 0 && f.n <= kMaxRaysPerFrame && f.src >= 0);
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    double qa_lo = inf, qa_hi = -inf, qb_lo = inf, qb_hi = -inf;
    for (int j = threadIdx.x; j < kMaxRaysPerFrame; j += kIngestThreads) {
        s_idx[j] = j;
        if (j >= f.n) s_ts[j] = inf;  // padding sorts last (a slot >= n is never a caller index)
    }
    for (int j = threadIdx.x; j < f.n; j += kIngestThreads) {  // stored slot j holds caller ray i
        const int i = src_orig[f.src + j];
        RS_ASSERT(i >= 0 && i < f.n);
        const double* t = src_rays + ((size_t)f.src + (j & ~31)) * 8 + (j & 31);
        const double2 q = rowq[f.src + i];
        s_ts[i] = f.ts_a + ro * q.x;      // ingest_pixels_kernel's (core_testcode.cpp:144)
        s_val[0][i] = f.ts_b + ro * q.y;  // (:145)
#pragma unroll
        for (int c = 1; c < 7; ++c) s_val[c][i] = t[32 * (c + 1)];
        qa_lo = fmin(qa_lo, q.x); qa_hi = fmax(qa_hi, q.x);
        qb_lo = fmin(qb_lo, q.y); qb_hi = fmax(qb_hi, q.y);
    }
    if (ext) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            qa_lo = fmin(qa_lo, __shfl_xor_sync(FULL, qa_lo, o)); qa_hi = fmax(qa_hi, __shfl_xor_sync(FULL, qa_hi, o));
            qb_lo = fmin(qb_lo, __shfl_xor_sync(FULL, qb_lo, o)); qb_hi = fmax(qb_hi, __shfl_xor_sync(FULL, qb_hi, o));
        }
        if ((threadIdx.x & 31) == 0) {
            double* e = s_ext[threadIdx.x >> 5];
            e[0] = qa_lo; e[1] = qa_hi; e[2] = qb_lo; e[3] = qb_hi;
        }
    }
    __syncthreads();  // the whole frame is staged: from here on the block may overwrite its source
    if (ext && threadIdx.x == 0) {
        for (int w = 1; w < kIngestThreads / 32; ++w) {
            qa_lo = fmin(qa_lo, s_ext[w][0]); qa_hi = fmax(qa_hi, s_ext[w][1]);
            qb_lo = fmin(qb_lo, s_ext[w][2]); qb_hi = fmax(qb_hi, s_ext[w][3]);
        }
        ext[blockIdx.x] = make_double4(qa_lo, qa_hi, qb_lo, qb_hi);
    }
    ingest_sort_and_store(f, s_ts, s_idx, s_val, rays, orig, pos);
}

// the same with the rays already computed by the caller (SetTrackResult's layouts).
// kRowFractions: the ts slots hold row fractions q instead; ts = frame_ts + ro * q with
// ingest_pixels_kernel's expression (PixelFrame::ts_a / ts_b), and q is kept in rowq for re-timing.
template <bool kRowFractions>
__global__ void __launch_bounds__(kIngestThreads)
ingest_rays_kernel(const PixelFrame* __restrict__ frames, const double* __restrict__ ts_a,
                   const double* __restrict__ ts_b, const double* __restrict__ ra,
                   const double* __restrict__ rb, double ro, double* __restrict__ rays, int32_t* __restrict__ orig,
                   int32_t* __restrict__ pos, double2* __restrict__ rowq) {
    __shared__ double s_ts[kMaxRaysPerFrame];
    __shared__ int s_idx[kMaxRaysPerFrame];
    __shared__ double s_val[7][kMaxRaysPerFrame];
    const PixelFrame f = frames[blockIdx.x];
    for (int i = threadIdx.x; i < kMaxRaysPerFrame; i += kIngestThreads) {
        s_idx[i] = i;
        if (i < f.n) {
            const size_t g = (size_t)f.src + i;
            if (kRowFractions) {
                const double qa = ts_a[g], qb = ts_b[g];
                rowq[f.off + i] = make_double2(qa, qb);
                s_ts[i] = f.ts_a + ro * qa;
                s_val[0][i] = f.ts_b + ro * qb;
            } else {
                s_ts[i] = ts_a[g];
                s_val[0][i] = ts_b[g];
            }
            s_val[1][i] = ra[3 * g]; s_val[2][i] = ra[3 * g + 1]; s_val[3][i] = ra[3 * g + 2];
            s_val[4][i] = rb[3 * g]; s_val[5][i] = rb[3 * g + 1]; s_val[6][i] = rb[3 * g + 2];
        } else {
            s_ts[i] = __longlong_as_double(0x7ff0000000000000LL);
        }
    }
    __syncthreads();
    ingest_sort_and_store(f, s_ts, s_idx, s_val, rays, orig, pos);
}

// Check-and-stage of track buffers that already live in device memory (the host's stage_track pass,
// capi.cpp, on the device).  One block per frame; each source buffer's segment of the frame is
// contiguous, so the block reads it once, coalesced, and writes it to the staging buffer at the same
// offset.  Per frame: which buffers hold a NaN / infinity, and the timestamp bounds.  Copies and
// comparisons only (pixels and row-fractions forms: plus ingest_pixels_kernel's timestamp expression,
// the same IEEE operations as the host's), so the bounds are the host form's values.  Only 8-byte
// alignment of the sources is assumed (a tensor view may start at any element).
constexpr int kStageThreads = 128;
struct StageArgs {
    const int64_t* at;  // n_frames + 1 offsets, in rays
    int64_t total;
    const double* src[4];
    double* dst[4];
    const double* frame_ts;  // pixels and row-fractions forms: ts_a, ts_b per frame
    double ro, rows;
    StageInfo* info;
    double fx, fy, cx, cy;  // pixels form: the lens's normalisation (undistort_point)
};
enum class StageMode { kRays, kPoints, kRowFractions };
template <StageMode M>
__global__ void __launch_bounds__(kStageThreads) stage_tracks_kernel(StageArgs a) {
    constexpr bool kPixels = M == StageMode::kPoints, kRowFractions = M == StageMode::kRowFractions;
    constexpr int NB = kPixels ? 2 : 4;
    const int f = blockIdx.x;
    const int64_t a0 = a.at[f], n = a.at[f + 1] - a0;
    RS_ASSERT(a0 >= 0 && n >= 0 && n <= kMaxRaysPerFrame && a0 + n <= a.total);
    unsigned bad = 0;
    double lo = __longlong_as_double(0x7ff0000000000000LL), hi = -lo;
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const int w = kPixels ? 2 : (b < 2 ? 3 : 1);  // doubles per ray
        const int64_t base = a0 * w, len = n * w;
        const double* __restrict__ s = a.src[b];
        double* __restrict__ d = a.dst[b];
        const double fts = kPixels                      ? a.frame_ts[2 * (int64_t)f + b]
                           : (kRowFractions && b >= 2) ? a.frame_ts[2 * (int64_t)f + (b - 2)]
                                                       : 0.0;
        for (int64_t j = threadIdx.x; j < len; j += kStageThreads) {
            RS_ASSERT(base + j < a.total * w);
            const double v = s[base + j];
            d[base + j] = v;
            if (!isfinite(v)) bad |= 1u << b;
            if (kPixels ? (j & 1) != 0 : b >= 2) {
                // (core_testcode.cpp:144-145); a row fraction whose timestamp overflows is as bad as a
                // non-finite one
                const double t = kPixels ? fts + a.ro * (v / a.rows) : kRowFractions ? fts + a.ro * v : v;
                if (kRowFractions && !isfinite(t)) bad |= 1u << b;
                // a finite point whose x_, y_ or theta_^2 in undistort_point overflows: its ray would be
                // NaN (the x of the point is the element before, read by the neighbouring lane)
                if (kPixels) {
                    const double x_ = (s[base + j - 1] - a.cx) / a.fx, y_ = (v - a.cy) / a.fy;
                    if (!isfinite(x_ * x_ + y_ * y_)) bad |= 1u << b;
                }
                lo = t < lo ? t : lo;
                hi = t > hi ? t : hi;
            }
        }
    }
    bad = __reduce_or_sync(FULL, bad);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double l = __shfl_xor_sync(FULL, lo, o), h = __shfl_xor_sync(FULL, hi, o);
        lo = l < lo ? l : lo;
        hi = h > hi ? h : hi;
    }
    constexpr int W = kStageThreads / 32;
    __shared__ unsigned s_bad[W];
    __shared__ double s_lo[W], s_hi[W];
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        RS_ASSERT(warp < W);
        s_bad[warp] = bad;
        s_lo[warp] = lo;
        s_hi[warp] = hi;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < W; ++k) {
            bad |= s_bad[k];
            lo = s_lo[k] < lo ? s_lo[k] : lo;
            hi = s_hi[k] > hi ? s_hi[k] : hi;
        }
        a.info[f] = StageInfo{bad, 0u, n ? lo : 0.0, n ? hi : 0.0};
    }
}

// ------------------------------------------------------------------------------------------
// Sparse pyramidal Lucas-Kanade (rssync_track_frames_device; the arithmetic contract is stated in
// include/rssync_b200.h).  The build uses -fmad=false, so every float32 expression below is evaluated
// in the order written.
struct TrackPyr {
    TrackImages im;
    float* lvl[kTrackMaxLevels];  // levels 1..: row y of slot s at lvl[l] + (s * h[l] + y) * w[l]
    int w[kTrackMaxLevels], h[kTrackMaxLevels];
    int slots;
    float scale;  // 2^-im.shift (a kernel parameter, so the 16-bit reads take it from the constant bank)
};

__device__ __forceinline__ int reflect101(int i, int n) {
    i = i < 0 ? -i : i;
    i = i >= n ? 2 * (n - 1) - i : i;
    return min(max(i, 0), n - 1);  // (only tile cells no output reads fall outside after the reflection)
}

// The level-0 intensity of a sample: (float)v, and for 16-bit samples (float)v * scale, scale = 2^-shift;
// both are exact (v < 2^16), so v = P << shift gives the 8-bit plane P's intensities bit for bit.
template <typename T>
__device__ __forceinline__ float track_level0(T v, float scale) {
    if constexpr (sizeof(T) == 1) return (float)v;
    else return (float)v * scale;
}

// level l of image j (slot j % slots above level 0) at integer (x, y), clamped to the level's edge
template <typename T>
__device__ __forceinline__ float track_px(const TrackPyr& P, int l, int j, int x, int y) {
    x = min(max(x, 0), P.w[l] - 1);
    y = min(max(y, 0), P.h[l] - 1);
    if (l == 0) {
        const T* row = reinterpret_cast<const T*>(P.im.img0 + ((int64_t)j * P.im.h0 + y) * P.im.pitch0);
        return track_level0<T>(__ldg(row + x), P.scale);
    }
    return __ldg(P.lvl[l] + ((int64_t)(j % P.slots) * P.h[l] + y) * P.w[l] + x);
}

template <typename T>
__device__ __forceinline__ float track_bilinear(const TrackPyr& P, int l, int j, int x, int y, float ax, float ay) {
    const float i00 = track_px<T>(P, l, j, x, y), i01 = track_px<T>(P, l, j, x + 1, y);
    const float i10 = track_px<T>(P, l, j, x, y + 1), i11 = track_px<T>(P, l, j, x + 1, y + 1);
    return (1.f - ay) * ((1.f - ax) * i00 + ax * i01) + ay * ((1.f - ax) * i10 + ax * i11);
}

// One launch per level: level l -> l + 1 of images [j0, j0 + gridDim.z).  A block's 32 x 8 outputs read a
// (2*8 + 3) x (2*32 + 3) tile of level l (BORDER_REFLECT_101), blur its rows into shared memory, then
// its columns: h = (s[-2] + s[2]) + 4 (s[-1] + s[1]) + 6 s[0] per row, the same over h per column, times
// 1/256.
// T: the type of the level-0 samples (uint8_t or uint16_t).
constexpr int kPyrTX = 32, kPyrTY = 8;
template <typename T>
__global__ void __launch_bounds__(kPyrTX * kPyrTY) track_pyramid_kernel(TrackPyr P, int l, int j0) {
    constexpr int TH = 2 * kPyrTY + 3, TW = 2 * kPyrTX + 3;
    __shared__ float s_in[TH][TW];
    __shared__ float s_h[TH][kPyrTX];
    const int j = j0 + blockIdx.z;
    const int w = P.w[l], h = P.h[l];
    const int X0 = blockIdx.x * kPyrTX, Y0 = blockIdx.y * kPyrTY;
    for (int k = threadIdx.x; k < TH * TW; k += kPyrTX * kPyrTY) {
        const int r = k / TW, c = k % TW;
        s_in[r][c] = track_px<T>(P, l, j, reflect101(2 * X0 - 2 + c, w), reflect101(2 * Y0 - 2 + r, h));
    }
    __syncthreads();
    for (int k = threadIdx.x; k < TH * kPyrTX; k += kPyrTX * kPyrTY) {
        const int r = k / kPyrTX, c = k % kPyrTX;
        const float* s = &s_in[r][2 * c];
        s_h[r][c] = ((s[0] + s[4]) + 4.f * (s[1] + s[3])) + 6.f * s[2];
    }
    __syncthreads();
    const int tx = threadIdx.x % kPyrTX, ty = threadIdx.x / kPyrTX;
    const int X = X0 + tx, Y = Y0 + ty;
    if (X < P.w[l + 1] && Y < P.h[l + 1]) {
        const int r = 2 * ty;
        const float v = ((s_h[r][tx] + s_h[r + 4][tx]) + 4.f * (s_h[r + 1][tx] + s_h[r + 3][tx])) + 6.f * s_h[r + 2][tx];
        P.lvl[l + 1][((int64_t)(j % P.slots) * P.h[l + 1] + Y) * P.w[l + 1] + X] = v * (1.f / 256.f);
    }
}

// Eligibility planes of the caller's mask (rssync_track_frames_masked_device): image j's byte of pixel
// (x, y) at plane + (j % slots) * stride + y * w0 + x, 1 = eligible (stride 0: one plane for every image).
// The unmasked kernels take it as their last parameter and never read it, so their other parameters keep
// their offsets.
struct TrackElig {
    const uint8_t* plane;
    int64_t stride;
    int slots;
};

// whether the position (x, y) of image j is eligible, looked up at its nearest pixel (floor(x + 0.5),
// floor(y + 0.5)); (x, y) lies in [0, w0 - 1] x [0, h0 - 1]
__device__ __forceinline__ bool track_eligible(const TrackElig& E, int w0, int j, double x, double y) {
    const int ix = (int)floor(x + 0.5), iy = (int)floor(y + 0.5);
    return E.plane[(int64_t)(j % E.slots) * E.stride + (int64_t)iy * w0 + ix] != 0;
}

// Erosion of images [j0, j0 + gridDim.z) of the mask by a (2 m + 1)^2 square (cv2.erode of mask != 0, pixels
// outside the image usable): a block's kErTX x kErTY outputs read a (kErTY + 2m) x (kErTX + 2m) tile, AND
// its rows over 2m + 1 columns into shared memory, then the columns over 2m + 1 rows.
constexpr int kErTX = 64, kErTY = 32;
__global__ void __launch_bounds__(256) track_erode_kernel(TrackMask M, int w, int h, int j0, TrackElig E) {
    constexpr int MH = kErTY + 2 * kTrackMaxMargin, MW = kErTX + 2 * kTrackMaxMargin;
    __shared__ uint8_t s_in[MH][MW];
    __shared__ uint8_t s_row[MH][kErTX];
    const int m = M.margin, th = kErTY + 2 * m, tw = kErTX + 2 * m;
    const int j = j0 + blockIdx.z;
    const int X0 = blockIdx.x * kErTX - m, Y0 = blockIdx.y * kErTY - m;
    const uint8_t* mask = M.mask + (int64_t)j * M.image_stride;
    for (int k = threadIdx.x; k < th * tw; k += blockDim.x) {
        const int r = k / tw, c = k % tw, x = X0 + c, y = Y0 + r;
        s_in[r][c] = x < 0 || x >= w || y < 0 || y >= h || mask[(int64_t)y * M.pitch + x] != 0;
    }
    __syncthreads();
    for (int k = threadIdx.x; k < th * kErTX; k += blockDim.x) {
        const int r = k / kErTX, c = k % kErTX;
        uint8_t v = 1;
        for (int i = 0; i <= 2 * m; ++i) v &= s_in[r][c + i];
        s_row[r][c] = v;
    }
    __syncthreads();
    uint8_t* out = const_cast<uint8_t*>(E.plane) + (int64_t)(j % E.slots) * E.stride;
    for (int k = threadIdx.x; k < kErTY * kErTX; k += blockDim.x) {
        const int r = k / kErTX, c = k % kErTX, x = X0 + m + c, y = Y0 + m + r;
        if (x >= w || y >= h) continue;
        uint8_t v = 1;
        for (int i = 0; i <= 2 * m; ++i) v &= s_row[r + i][c];
        out[(int64_t)y * w + x] = v;
    }
}

// sum over the 32 lanes: xor butterfly 16, 8, 4, 2, 1 (every lane ends with the same bits)
__device__ __forceinline__ float track_warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// One warp per query point, all levels.  Per warp in shared memory: the side-a patch, (window + 2)^2
// bilinear samples, and its Scharr gradients over the window.
// kBack: the backward pass of the forward-backward check.  Only points with status 1 take part; the
// query is the forward result tracked[k] on image i + 1 (side a), side b is image i; the result u gives
// fb = |u - pts[k]| (double) in fb_out[k] when u is kept (lost: fb_out[k] keeps the NaN it was filled
// with), and the status becomes 2 unless u is kept and fb <= fb_max.
// The forward instantiation writes neither fb_out nor reads fb_max.
// kMask (forward only): a point kept forward gets status 3 instead of 1 when its query position is not
// eligible on image i or its tracked position is not eligible on image i + 1 (E).
constexpr int kLkWarps = 4;
// Minimum blocks per SM in the launch bounds: 0 (none) for 8-bit samples; 7 (at most 72 registers) for
// 16-bit samples, which ptxas otherwise fits in 64 registers with a spill.
template <typename T>
constexpr int kLkMinBlocks = sizeof(T) == 1 ? 0 : 7;
template <typename T, bool kBack, bool kMask = false>
__global__ void __launch_bounds__(kLkWarps * 32, kLkMinBlocks<T>)
    track_lk_kernel(TrackPyr P, const int64_t* __restrict__ q_at, int f0, int f1, const double* __restrict__ pts,
                    double* __restrict__ tracked, uint8_t* __restrict__ status, unsigned* flag, double fb_max,
                    double* __restrict__ fb_out, TrackElig E) {
    static_assert(!(kBack && kMask), "the backward pass runs on status 1 only and takes no mask");
    extern __shared__ float s_lk[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int win = P.im.window, r = win / 2, pw = win + 2, nw = win * win;
    float* sA = s_lk + (size_t)warp * (pw * pw + 2 * nw);
    float* sIx = sA + pw * pw;
    float* sIy = sIx + nw;
    const int64_t k = q_at[f0] + (int64_t)blockIdx.x * kLkWarps + warp;
    if (k >= q_at[f1]) return;
    int lo = f0, hi = f1 - 1;  // the frame holding point k: the last f with q_at[f] <= k
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (q_at[mid] <= k) lo = mid; else hi = mid - 1;
    }
    const int ja = kBack ? lo + 1 : lo, jb = kBack ? lo : lo + 1;
    if (kBack && status[k] != 1) return;
    const double qx = kBack ? tracked[2 * k] : pts[2 * k], qy = kBack ? tracked[2 * k + 1] : pts[2 * k + 1];
    const bool finite = isfinite(qx) && isfinite(qy);
    if (!kBack && !finite && lane == 0) atomicOr(flag, 1u);
    bool ok = finite && qx >= 0.0 && qx <= P.w[0] - 1 && qy >= 0.0 && qy <= P.h[0] - 1;
    const float px0 = (float)qx, py0 = (float)qy;
    const float eps2 = P.im.epsilon * P.im.epsilon, area = (float)nw;
    float gx = 0.f, gy = 0.f, vx = 0.f, vy = 0.f;
    for (int l = P.im.levels - 1; ok && l >= 0; --l) {
        const float s = ldexpf(1.f, -l);
        const float ax = px0 * s, ay = py0 * s;
        const float fx = floorf(ax), fy = floorf(ay);
        const float wx = ax - fx, wy = ay - fy;
        const int ix = (int)fx, iy = (int)fy;
        __syncwarp();  // the previous level's readers of sA are done
        for (int t = lane; t < pw * pw; t += 32)
            sA[t] = track_bilinear<T>(P, l, ja, ix + t % pw - r - 1, iy + t / pw - r - 1, wx, wy);
        __syncwarp();
        float gxx = 0.f, gxy = 0.f, gyy = 0.f;
        for (int t = lane; t < nw; t += 32) {
            const float* c = sA + (t / win + 1) * pw + (t % win + 1);
            const float dx = ((3.f * (c[-pw + 1] - c[-pw - 1]) + 10.f * (c[1] - c[-1])) + 3.f * (c[pw + 1] - c[pw - 1])) *
                             (1.f / 32.f);
            const float dy = ((3.f * (c[pw - 1] - c[-pw - 1]) + 10.f * (c[pw] - c[-pw])) + 3.f * (c[pw + 1] - c[-pw + 1])) *
                             (1.f / 32.f);
            sIx[t] = dx;
            sIy[t] = dy;
            gxx += dx * dx;
            gxy += dx * dy;
            gyy += dy * dy;
        }
        gxx = track_warp_sum(gxx);
        gxy = track_warp_sum(gxy);
        gyy = track_warp_sum(gyy);
        const float d = gxx - gyy;
        const float min_eig = ((gxx + gyy) - sqrtf(d * d + 4.f * (gxy * gxy))) / (2.f * area);
        if (!(min_eig >= P.im.min_eig)) { ok = false; break; }
        const float det = gxx * gyy - gxy * gxy;
        __syncwarp();
        // side b positions far outside the level read its edge pixels only: clamp them there first so the
        // integer conversion stays in range
        const float lim_lo = -2.f * pw, lim_x = (float)(P.w[l] + 2 * pw), lim_y = (float)(P.h[l] + 2 * pw);
        for (int it = 0; it < P.im.max_iters; ++it) {
            const float bxp = ax + gx + vx, byp = ay + gy + vy;
            const float bfx = floorf(bxp), bfy = floorf(byp);
            const float bwx = bxp - bfx, bwy = byp - bfy;
            const int bix = (int)fminf(fmaxf(bfx, lim_lo), lim_x), biy = (int)fminf(fmaxf(bfy, lim_lo), lim_y);
            float bx = 0.f, by = 0.f;
            for (int t = lane; t < nw; t += 32) {
                const int tx = t % win, ty = t / win;
                const float B = track_bilinear<T>(P, l, jb, bix + tx - r, biy + ty - r, bwx, bwy);
                const float diff = sA[(ty + 1) * pw + tx + 1] - B;
                bx += diff * sIx[t];
                by += diff * sIy[t];
            }
            bx = track_warp_sum(bx);
            by = track_warp_sum(by);
            const float ex = (gyy * bx - gxy * by) / det, ey = (gxx * by - gxy * bx) / det;
            if (!isfinite(ex) || !isfinite(ey)) { ok = false; break; }
            vx += ex;
            vy += ey;
            if (ex * ex + ey * ey < eps2) break;
        }
        if (!ok) break;
        if (l > 0) {
            gx = 2.f * (gx + vx);
            gy = 2.f * (gy + vy);
            vx = vy = 0.f;
        }
    }
    if (lane == 0) {
        double tx = __longlong_as_double(0x7ff8000000000000LL), ty = tx;  // NaN: lost before the last level ended
        if (ok) {
            tx = qx + (double)(gx + vx);
            ty = qy + (double)(gy + vy);
            ok = tx >= 0.0 && tx <= P.w[0] - 1 && ty >= 0.0 && ty <= P.h[0] - 1;
        }
        if constexpr (kBack) {
            const double ex = tx - pts[2 * k], ey = ty - pts[2 * k + 1];
            const double fb = sqrt(ex * ex + ey * ey);
            if (ok && fb_out) fb_out[k] = fb;  // (the caller filled fb_out with NaN)
            status[k] = ok && fb <= fb_max ? 1 : 2;
        } else {
            tracked[2 * k] = tx;
            tracked[2 * k + 1] = ty;
            if constexpr (kMask)
                status[k] = !ok ? 0
                            : track_eligible(E, P.w[0], lo, qx, qy) && track_eligible(E, P.w[0], lo + 1, tx, ty) ? 1
                                                                                                                : 3;
            else
                status[k] = ok ? 1 : 0;
        }
    }
}

// One block: kept count per frame (warp per frame), prefix sum (warp 0), then every warp writes its
// frames' kept pairs in query order.
constexpr int kCompactThreads = 1024;
__global__ void __launch_bounds__(kCompactThreads) track_compact_kernel(const int64_t* __restrict__ q_at, int n,
                                                                       const double* __restrict__ pts,
                                                                       const double* __restrict__ tracked,
                                                                       const uint8_t* __restrict__ status,
                                                                       double* __restrict__ out_a,
                                                                       double* __restrict__ out_b, int64_t* kept_at) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int W = kCompactThreads / 32;
    for (int f = warp; f < n; f += W) {
        int64_t c = 0;
        for (int64_t k = q_at[f] + lane; k - lane < q_at[f + 1]; k += 32)
            c += __popc(__ballot_sync(FULL, k < q_at[f + 1] && status[k] == 1));
        if (lane == 0) kept_at[f + 1] = c;
    }
    __syncthreads();
    if (warp == 0) {
        int64_t carry = 0;
        if (lane == 0) kept_at[0] = 0;
        for (int base = 0; base < n; base += 32) {
            int64_t v = base + lane < n ? kept_at[base + lane + 1] : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int64_t u = __shfl_up_sync(FULL, v, o);
                if (lane >= o) v += u;
            }
            v += carry;
            if (base + lane < n) kept_at[base + lane + 1] = v;
            carry = __shfl_sync(FULL, v, 31);
        }
    }
    __syncthreads();
    for (int f = warp; f < n; f += W) {
        int64_t o = kept_at[f];
        for (int64_t k = q_at[f] + lane; k - lane < q_at[f + 1]; k += 32) {
            const bool keep = k < q_at[f + 1] && status[k] == 1;
            const unsigned m = __ballot_sync(FULL, keep);
            if (keep) {
                const int64_t d = o + __popc(m & ((1u << lane) - 1u));
                out_a[2 * d] = pts[2 * k];
                out_a[2 * d + 1] = pts[2 * k + 1];
                out_b[2 * d] = tracked[2 * k];
                out_b[2 * d + 1] = tracked[2 * k + 1];
            }
            o += __popc(m);
        }
    }
}

// ------------------------------------------------------------------------------------------
// Point selection (rssync_track_frames_ex_device; the contract is stated in include/rssync_b200.h):
// the minimum eigenvalue of the structure tensor (cv2.cornerMinEigenVal), its 3 x 3 local maxima, the
// best of each cell, then a threshold and a top-max_points cut per image.  float32 in the order written
// (-fmad=false), so the scores equal a numpy float32 restatement bit for bit.
constexpr int kSelThreads = 256, kSelStrip = 32, kPickThreads = 1024;

// One block per (cell, image).  Shared memory: the cell's pixels with a halo of block / 2 + 2, the
// scores of the cell and a 1-pixel ring, and, per strip of kSelStrip score rows, the Sobel gradients
// and the row sums of their products.  The halo keeps every pixel a candidate's or its neighbours'
// scores read inside the image, so reads outside it (clamped here) reach no used score.  Writes the
// cell's best candidate as the key (score bits << 32) | ~(y * w + x): the greater key is the greater
// score, then the smaller index; 0 = no candidate.  The pixels are staged as the plane's samples (T) and
// converted by track_level0 where the Sobel stencil reads them.  kMask: a candidate must also be eligible (E).
template <typename T, bool kMask = false>
__global__ void __launch_bounds__(kSelThreads) select_cells_kernel(TrackImages im, TrackSelect S, int j0, TrackElig E) {
    extern __shared__ float s_sel[];
    const int C = S.cell, B = S.block, r = B / 2, hal = r + 2;
    const int PW = C + 2 * hal, SW = C + 2, GW = SW + 2 * r, GR = kSelStrip + 2 * r;
    float* sS = s_sel;           // SW x SW scores: row sy, column sx <-> (X0 - 1 + sx, Y0 - 1 + sy)
    float* sDx = sS + SW * SW;   // GR x GW gradients of a strip
    float* sDy = sDx + GR * GW;
    float* sHxx = sDy + GR * GW;  // GR x SW row sums of a strip
    float* sHxy = sHxx + GR * SW;
    float* sHyy = sHxy + GR * SW;
    T* sP = reinterpret_cast<T*>(sHyy + GR * SW);  // PW x PW samples from (X0 - hal, Y0 - hal)
    const int w = im.w0, h = im.h0;
    const int X0 = (blockIdx.x % S.cells_x) * C, Y0 = (blockIdx.x / S.cells_x) * C;
    const uint8_t* img = im.img0 + (int64_t)(j0 + blockIdx.y) * h * im.pitch0;
    for (int t = threadIdx.x; t < PW * PW; t += kSelThreads) {
        const int y = min(max(Y0 - hal + t / PW, 0), h - 1), x = min(max(X0 - hal + t % PW, 0), w - 1);
        sP[t] = __ldg(reinterpret_cast<const T*>(img + (int64_t)y * im.pitch0) + x);
    }
    const float sc = (float)(1.0 / (4.0 * B * 255.0)), scale = ldexpf(1.f, -im.shift);
    __syncthreads();
    for (int s0 = 0; s0 < SW; s0 += kSelStrip) {
        const int nr = min(kSelStrip, SW - s0), gr = nr + 2 * r;
        // gradient row t, column u <-> (X0 - 1 - r + u, Y0 - 1 - r + s0 + t), pixel row s0 + t + 1, column u + 1
        for (int t = threadIdx.x; t < gr * GW; t += kSelThreads) {
            const T* c = sP + (s0 + t / GW + 1) * PW + t % GW + 1;
            const float i00 = track_level0<T>(c[-PW - 1], scale), i01 = track_level0<T>(c[-PW], scale);
            const float i02 = track_level0<T>(c[-PW + 1], scale), i10 = track_level0<T>(c[-1], scale);
            const float i12 = track_level0<T>(c[1], scale), i20 = track_level0<T>(c[PW - 1], scale);
            const float i21 = track_level0<T>(c[PW], scale), i22 = track_level0<T>(c[PW + 1], scale);
            sDx[t] = (((i02 - i00) + 2.f * (i12 - i10)) + (i22 - i20)) * sc;
            sDy[t] = (((i20 - i00) + 2.f * (i21 - i01)) + (i22 - i02)) * sc;
        }
        __syncthreads();
        // row sums: column v <-> x = X0 - 1 + v adds gradient columns v .. v + 2r, left to right
        for (int t = threadIdx.x; t < gr * SW; t += kSelThreads) {
            const float* dx = sDx + (t / SW) * GW + t % SW;
            const float* dy = sDy + (t / SW) * GW + t % SW;
            float xx = dx[0] * dx[0], xy = dx[0] * dy[0], yy = dy[0] * dy[0];
            for (int i = 1; i < B; ++i) {
                xx += dx[i] * dx[i];
                xy += dx[i] * dy[i];
                yy += dy[i] * dy[i];
            }
            sHxx[t] = xx;
            sHxy[t] = xy;
            sHyy[t] = yy;
        }
        __syncthreads();
        // score row s0 + t adds row sums t .. t + 2r, top to bottom
        for (int t = threadIdx.x; t < nr * SW; t += kSelThreads) {
            float xx = sHxx[t], xy = sHxy[t], yy = sHyy[t];
            for (int i = 1; i < B; ++i) {
                xx += sHxx[t + i * SW];
                xy += sHxy[t + i * SW];
                yy += sHyy[t + i * SW];
            }
            const float a = 0.5f * xx, c = 0.5f * yy, d = a - c;
            sS[s0 * SW + t] = (a + c) - sqrtf(d * d + xy * xy);
        }
        __syncthreads();
    }
    const int m = hal;
    unsigned long long best = 0;
    for (int t = threadIdx.x; t < C * C; t += kSelThreads) {
        const int x = X0 + t % C, y = Y0 + t / C;
        if (x < m || x > w - 1 - m || y < m || y > h - 1 - m) continue;
        const float* c = sS + (t / C + 1) * SW + t % C + 1;
        const float v = c[0];
        if (v > 0.f && v >= c[-SW - 1] && v >= c[-SW] && v >= c[-SW + 1] && v >= c[-1] && v >= c[1] &&
            v >= c[SW - 1] && v >= c[SW] && v >= c[SW + 1]) {
            // (read for the local maxima only: a load per pixel of the cell would stall this loop)
            if constexpr (kMask)
                if (!E.plane[(int64_t)((j0 + blockIdx.y) % E.slots) * E.stride + (int64_t)y * w + x]) continue;
            const unsigned long long key = ((unsigned long long)__float_as_uint(v) << 32) |
                                           (unsigned)~((unsigned)y * (unsigned)w + (unsigned)x);
            best = key > best ? key : best;
        }
    }
    __shared__ unsigned long long s_best[kSelThreads / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long u = __shfl_xor_sync(FULL, best, o);
        best = u > best ? u : best;
    }
    if ((threadIdx.x & 31) == 0) s_best[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < kSelThreads / 32; ++i) best = s_best[i] > best ? s_best[i] : best;
        S.d_keys[(size_t)blockIdx.y * S.cells_x * S.cells_y + blockIdx.x] = best;
    }
}

__device__ __forceinline__ unsigned block_reduce_max_sum(unsigned v, bool is_max, unsigned* s_red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned u = __shfl_xor_sync(FULL, v, o);
        v = is_max ? max(v, u) : v + u;
    }
    __syncthreads();  // (s_red's previous readers are done)
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    v = s_red[0];
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i) v = is_max ? max(v, s_red[i]) : v + s_red[i];
    return v;
}

// One block per image of a chunk: M (the greatest pick score), the threshold (float)quality * M, and,
// when more than max_points picks pass it, the max_points-th greatest selection key (score bits << 32) |
// ~cell by an MSB radix select (8 passes of 8 bits; the keys are distinct).  Then the kept picks in
// ascending cell order: their pixel indices to d_picks[image * max_points ..], their number to d_count.
__global__ void __launch_bounds__(kPickThreads) select_points_kernel(TrackSelect S) {
    __shared__ unsigned s_red[kPickThreads / 32];
    __shared__ unsigned s_hist[256];
    __shared__ unsigned long long s_cut;
    __shared__ unsigned s_need;
    const int nc = S.cells_x * S.cells_y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long* keys = S.d_keys + (size_t)blockIdx.x * nc;
    unsigned mx = 0;
    for (int c = threadIdx.x; c < nc; c += kPickThreads) mx = max(mx, (unsigned)(keys[c] >> 32));
    mx = block_reduce_max_sum(mx, true, s_red);
    const float thr = S.quality * __uint_as_float(mx);
    auto kept = [&](unsigned long long key) { return key != 0 && __uint_as_float((unsigned)(key >> 32)) >= thr; };
    unsigned n = 0;
    for (int c = threadIdx.x; c < nc; c += kPickThreads) n += kept(keys[c]) ? 1u : 0u;
    n = block_reduce_max_sum(n, false, s_red);
    unsigned long long cut = 0;  // keep a pick whose selection key is >= cut
    if (n > (unsigned)S.max_points) {
        if (threadIdx.x == 0) {
            s_cut = 0;
            s_need = S.max_points;
        }
        for (int shift = 56; shift >= 0; shift -= 8) {
            for (int i = threadIdx.x; i < 256; i += kPickThreads) s_hist[i] = 0;
            __syncthreads();
            const unsigned long long hi = shift == 56 ? 0ull : ~0ull << (shift + 8), pre = s_cut & hi;
            for (int c = threadIdx.x; c < nc; c += kPickThreads) {
                const unsigned long long key = keys[c];
                const unsigned long long sk = (key & 0xffffffff00000000ull) | (unsigned)~(unsigned)c;
                if (kept(key) && (sk & hi) == pre) atomicAdd(&s_hist[(sk >> shift) & 255], 1u);
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                unsigned need = s_need;
                int d = 255;
                for (; d > 0 && s_hist[d] < need; --d) need -= s_hist[d];
                s_need = need;
                s_cut |= (unsigned long long)d << shift;
            }
            __syncthreads();
        }
        cut = s_cut;
    }
    unsigned base = 0;
    for (int c0 = 0; c0 < nc; c0 += kPickThreads) {
        const int c = c0 + threadIdx.x;
        const unsigned long long key = c < nc ? keys[c] : 0ull;
        const bool keep = kept(key) && ((key & 0xffffffff00000000ull) | (unsigned)~(unsigned)c) >= cut;
        const unsigned bal = __ballot_sync(FULL, keep);
        __syncthreads();  // (s_red's previous readers are done)
        if (lane == 0) s_red[warp] = __popc(bal);
        __syncthreads();
        unsigned off = base, tot = 0;
        for (int i = 0; i < kPickThreads / 32; ++i) {
            off += i < warp ? s_red[i] : 0u;
            tot += s_red[i];
        }
        if (keep) S.d_picks[(size_t)blockIdx.x * S.max_points + off + __popc(bal & ((1u << lane) - 1u))] = ~(unsigned)key;
        base += tot;
    }
    if (threadIdx.x == 0) S.d_count[blockIdx.x] = (int32_t)base;
}

// One block: the prefix of the picks of frames [f0, f1) from q_at[f0] (q_at[0] = 0) into q_at, then
// every frame's picks as points ((double)x, (double)y) at their offsets.
__global__ void __launch_bounds__(kPickThreads) select_prefix_kernel(TrackSelect S, int64_t* q_at, int f0, int f1,
                                                                     int w, double* __restrict__ pts) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n = f1 - f0;
    constexpr int W = kPickThreads / 32;
    if (warp == 0) {
        int64_t carry = f0 == 0 ? 0 : q_at[f0];
        if (f0 == 0 && lane == 0) q_at[0] = 0;
        for (int base = 0; base < n; base += 32) {
            int64_t v = base + lane < n ? S.d_count[base + lane] : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int64_t u = __shfl_up_sync(FULL, v, o);
                if (lane >= o) v += u;
            }
            v += carry;
            if (base + lane < n) q_at[f0 + base + lane + 1] = v;
            carry = __shfl_sync(FULL, v, 31);
        }
    }
    __syncthreads();
    for (int i = warp; i < n; i += W) {
        const int64_t o = q_at[f0 + i];
        for (int k = lane; k < S.d_count[i]; k += 32) {
            const unsigned idx = S.d_picks[(size_t)i * S.max_points + k];
            pts[2 * (o + k)] = (double)(idx % (unsigned)w);
            pts[2 * (o + k) + 1] = (double)(idx / (unsigned)w);
        }
    }
}

// ------------------------------------------------------------------------------------------
// K7:the parallel half of ndspline::make (ndspline.cpp:13-19 / minispline.cpp:34-44).  The host
// eliminates the tridiagonal system (two sequential sweeps, host_ingest.cpp) and sends what is left
// of it -- rhs and diag, 5 doubles per sample instead of the 16 of a finished record -- with the
// samples themselves; one thread per (sample, component) divides (:34), forms b and d of the
// interval (:38-44, the reference's expressions; IEEE operations without contraction, so the bits
// of the host evaluation) and writes the record in the device's swizzled group order (rec_groups).
__global__ void spline_finish_kernel(const double* __restrict__ y, const double* __restrict__ rhs,
                                     const double* __restrict__ diag, int n, double* __restrict__ rec) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 4LL * n) return;
    const int i = (int)(t >> 2), c = (int)(t & 3);
    const double yi = y[4 * (size_t)i + c];
    const double ci = rhs[4 * (size_t)i + c] / diag[i];
    double b, d;
    if (i + 1 < n) {
        const double cn = rhs[4 * (size_t)(i + 1) + c] / diag[i + 1];
        d = 1.0 / 3.0 * (cn - ci);                                              // :40
        b = (y[4 * (size_t)(i + 1) + c] - yi) - 1.0 / 3.0 * (2.0 * ci + cn);   // :41
    } else {  // last sample (:43-44), from the coefficients of the interval before it
        const double cp = rhs[4 * (size_t)(i - 1) + c] / diag[i - 1];
        const double dp = 1.0 / 3.0 * (ci - cp);
        const double bp = (yi - y[4 * (size_t)(i - 1) + c]) - 1.0 / 3.0 * (2.0 * cp + ci);
        d = 0.0;
        b = (3.0 * dp + 2.0 * cp) + bp;
    }
    double* out = rec + (size_t)i * 16 + c;
    const int sw = (i & 3) * 4;
    out[0 ^ sw] = yi;
    out[4 ^ sw] = b;
    out[8 ^ sw] = ci;
    out[12 ^ sw] = d;
}

// ------------------------------------------------------------------------------------------
// K8: the gyro ingest on the device, for n_var gyro axis mappings (3x3 matrices, gyro_scan.h) at once.
//
//  * gyro_local / gyro_prefix / gyro_apply: optdata_fill_gyro (core_testcode.cpp:37-53) as a blocked
//    scan.  q_i = normalise(d_i (x) q_{i-1}) is not associative once every step normalises, so the
//    contract fixes the order (gyro_scan.h, shared with the host code and the oracle): the
//    recurrence inside blocks of kGyroScanBlock samples from the identity (one thread per block
//    and variant), the blocks' last values chained into prefixes (one thread per variant), then
//    every sample = normalise(local (x) prefix) in parallel.  sin / cos are the contract's
//    (spec_trig.h).
//  * resample: the per-sample half of the variable-rate SetGyroQuaternions (core_private.cpp:166-182):
//    grid point j = 1e6 (tick0 + j) / rate in integer division, lower_bound over the input
//    timestamps, quat_slerp (quat.cpp:55-74) with the contract's acos / sin; non-finite results raise
//    the variant's flag (:180).
//  * spline_chains: the two elimination sweeps of the spline system (minispline.cpp:22-32).  The
//    factors depend only on n (host_ingest.cpp); what is left per component is the first-order
//    recurrence rhs[i] -= rhs[i -+ 1] * f[i], sequential by nature: one thread per (variant,
//    component) walks it in the reference's order, so the bits are the host sweep's.  48 variants x 4
//    components run side by side, which is what the orientation search needs; a single long track is
//    faster on the host (SetGyroQuaternions' fixed-rate form keeps using it).
struct OrientDev {
    double m[9];  // the variant's gyro axis mapping, 3x3 row-major (gyro_scan.h)
};
__global__ void gyro_local_kernel(const double* __restrict__ ts, const double* __restrict__ gyro, int n,
                                  const OrientDev* __restrict__ orients, int n_var, double* __restrict__ local) {
    const int nb = (n + (int)kGyroScanBlock - 1) / (int)kGyroScanBlock;
    const int id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= nb * n_var) return;
    const int v = id / nb, b = id - v * nb;
    const OrientDev o = orients[v];
    double prev[4] = {1.0, 0.0, 0.0, 0.0};
    double* out = local + (size_t)v * n * 4;
    const int i1 = min(n, (b + 1) * (int)kGyroScanBlock);
    for (int i = b * (int)kGyroScanBlock; i < i1; ++i) {
        double d[4], q[4];
        gyro_increment(ts, gyro, (size_t)i, o.m, d);
        quat_mul_normalise(d, prev, q);
        prev[0] = q[0]; prev[1] = q[1]; prev[2] = q[2]; prev[3] = q[3];
        double2* dst = reinterpret_cast<double2*>(out + (size_t)i * 4);
        dst[0] = make_double2(q[0], q[1]);
        dst[1] = make_double2(q[2], q[3]);
    }
}
__global__ void gyro_prefix_kernel(const double* __restrict__ local, int n, int n_var, double* __restrict__ prefix) {
    const int nb = (n + (int)kGyroScanBlock - 1) / (int)kGyroScanBlock;
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_var) return;
    double* pf = prefix + (size_t)v * (nb + 1) * 4;
    double cur[4] = {1.0, 0.0, 0.0, 0.0};
    pf[0] = 1.0; pf[1] = 0.0; pf[2] = 0.0; pf[3] = 0.0;
    for (int b = 0; b < nb; ++b) {
        const int last = min(n, (b + 1) * (int)kGyroScanBlock) - 1;
        double nx[4];
        quat_mul_normalise(local + ((size_t)v * n + last) * 4, cur, nx);
        for (int c = 0; c < 4; ++c) { cur[c] = nx[c]; pf[(size_t)(b + 1) * 4 + c] = nx[c]; }
    }
}
__global__ void gyro_apply_kernel(const double* __restrict__ prefix, int n, int n_var, double* __restrict__ quats) {
    const int nb = (n + (int)kGyroScanBlock - 1) / (int)kGyroScanBlock;
    const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= (long long)n * n_var) return;
    const int v = (int)(id / n), i = (int)(id - (long long)v * n);
    double* q = quats + id * 4;  // in place: the block-local value becomes the sample
    const double loc[4] = {q[0], q[1], q[2], q[3]};
    double out[4];
    quat_mul_normalise(loc, prefix + ((size_t)v * (nb + 1) + i / (int)kGyroScanBlock) * 4, out);
    q[0] = out[0]; q[1] = out[1]; q[2] = out[2]; q[3] = out[3];
}
__global__ void resample_kernel(const int64_t* __restrict__ ts_us, int count, const double* __restrict__ quats,
                                int n_var, unsigned long long tick0, unsigned rate_hz, int n_out,
                                double* __restrict__ out, unsigned* __restrict__ nonfinite) {
    const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= (long long)n_out * n_var) return;
    const int v = (int)(id / n_out), j = (int)(id - (long long)v * n_out);
    const unsigned long long t = 1000000ULL * (tick0 + (unsigned long long)j) / rate_hz;  // core_private.cpp:153-154
    int lo = 0, hi = count;  // std::lower_bound: first index with ts_us[idx] >= t (as unsigned, :169)
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((unsigned long long)ts_us[mid] < t) lo = mid + 1; else hi = mid;
    }
    const double* src = quats + (size_t)v * count * 4;
    double r[4];
    if (lo > 0) {
        // lo < count: every grid point is below the last timestamp (plan_variable_rate)
        const double frac = 1. * (double)(t - (unsigned long long)ts_us[lo - 1]) / (double)(ts_us[lo] - ts_us[lo - 1]);
        quat_slerp_spec(src + (size_t)(lo - 1) * 4, src + (size_t)lo * 4, frac, r);  // :171-175
    } else {
        for (int c = 0; c < 4; ++c) r[c] = src[c];  // :177-178
    }
    double* dst = out + id * 4;
    dst[0] = r[0]; dst[1] = r[1]; dst[2] = r[2]; dst[3] = r[3];
    if (!(is_finite(r[0]) && is_finite(r[1]) && is_finite(r[2]) && is_finite(r[3]))) atomicOr(nonfinite + v, 1u);  // :180
}
__global__ void spline_chains_kernel(const double* __restrict__ y, const double* __restrict__ f_down,
                                     const double* __restrict__ f_up, int n, int n_var, double* __restrict__ rhs) {
    const int id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= 4 * n_var) return;
    const int v = id >> 2, c = id & 3;
    const double* q = y + (size_t)v * n * 4 + c;
    double* r = rhs + (size_t)v * n * 4 + c;
    r[0] = 0.0;
    r[(size_t)(n - 1) * 4] = 0.0;
    // The chains are dependent (one multiply and one subtraction per row); their operands are not:
    // U rows' worth of loads are issued before the U dependent steps that consume them, so the
    // memory latency is paid once per U rows instead of once per row.
    constexpr int U = 32;
    double prev = 0.0;  // rhs of row i - 1 after the downward sweep
    int i = 1;
    for (; i + U < n; i += U) {  // rows i .. i + U - 1, all interior (i + U - 1 + 1 < n)
        double qv[U + 2], fv[U];
#pragma unroll
        for (int k = 0; k < U + 2; ++k) qv[k] = q[(size_t)(i - 1 + k) * 4];
#pragma unroll
        for (int k = 0; k < U; ++k) fv[k] = f_down[i - 1 + k];
#pragma unroll
        for (int k = 0; k < U; ++k) {  // rhs of the row (:12-19) minus what the row above clears (:25)
            const double ri = (qv[k + 2] - 2 * qv[k + 1]) + qv[k];
            prev = ri - prev * fv[k];
            r[(size_t)(i + k) * 4] = prev;
        }
    }
    for (; i + 1 < n; ++i) {
        const double ri = (q[(size_t)(i + 1) * 4] - 2 * q[(size_t)i * 4]) + q[(size_t)(i - 1) * 4];
        prev = ri - prev * f_down[i - 1];
        r[(size_t)i * 4] = prev;
    }
    double nxt = 0.0;  // rhs of row i after the upward sweep (row n - 1: 0)
    i = n - 1;
    for (; i - U > 1; i -= U) {  // steps i, i - 1, ..., i - U + 1 write rows i - 1 ... i - U
        double rv[U], fv[U];
#pragma unroll
        for (int k = 0; k < U; ++k) rv[k] = r[(size_t)(i - 1 - k) * 4];
#pragma unroll
        for (int k = 0; k < U; ++k) fv[k] = f_up[i - k];
#pragma unroll
        for (int k = 0; k < U; ++k) {  // :31
            nxt = rv[k] - nxt * fv[k];
            r[(size_t)(i - 1 - k) * 4] = nxt;
        }
    }
    for (; i > 1; --i) {
        const double cur = r[(size_t)(i - 1) * 4] - nxt * f_up[i];
        r[(size_t)(i - 1) * 4] = cur;
        nxt = cur;
    }
}
__global__ void probe_trig_kernel(const double* __restrict__ x, int n, int which, double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = which == 0 ? spec_sin(x[i]) : which == 1 ? spec_cos(x[i]) : spec_acos(x[i]);
}

// ------------------------------------------------------------------------------------------
// probes (tests only): one warp
__global__ void probe_problem_kernel(DeviceData dd, FrameDesc fd, int NP, double delay, double* out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const WarpSmem w = warp_smem(smem_raw, 0, NP);
    build_rows_smem(dd, fd, delay, lane, w, NP);
    for (int i = lane; i < fd.n; i += 32) {  // back to the caller's ray order
        const int o = dd.orig[fd.off + i];
        out[3 * o] = w.P[i];
        out[3 * o + 1] = w.P[NP + i];
        out[3 * o + 2] = w.P[2 * NP + i];
    }
}
__global__ void probe_log1p_kernel(const double* x, int n, double* out) {
    __shared__ __align__(16) double tab[512];
    load_log1p_table(tab);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = log1p_nonneg(x[i], tab);
}
__global__ void probe_loss_kernel(DeviceData dd, FrameDesc fd, int NP, double delay, const double* mp,
                                  double k, double* out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    double* tab = reinterpret_cast<double*>(smem_raw);
    load_log1p_table(tab);
    const WarpSmem w = warp_smem(smem_raw + kLog1pTableBytes, 0, NP);
    const int nslots = (fd.n + 31) >> 5;
    build_rows_smem(dd, fd, delay, lane, w, NP);
    const double l3 = warp_loss3_smem(w.P, NP, nslots, lane, mp[0], mp[1], mp[2], k, tab);
    const Loss5 e = warp_loss5_smem(w.P, NP, nslots, lane, mp[0], mp[1], mp[2], k, tab);
    if (lane == 0) { out[0] = l3; out[1] = e.f; out[2] = e.g0; out[3] = e.g1; out[4] = e.g2; }
}
__global__ void probe_lbfgs_kernel(DeviceData dd, FrameDesc fd, int NP, double delay, double* mp,
                                   double k, double* fout, int* stats) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    double* tab = reinterpret_cast<double*>(smem_raw);
    load_log1p_table(tab);
    const WarpSmem w = warp_smem(smem_raw + kLog1pTableBytes, 0, NP);
    const int nslots = (fd.n + 31) >> 5;
    build_rows_smem(dd, fd, delay, lane, w, NP);
    double m[3] = {mp[0], mp[1], mp[2]};
    int it, ev;
    __shared__ double hist[kLbfgsHistDoubles];
    const double f = warp_lbfgs(
        [&](double a0, double a1, double a2) { return warp_loss5_smem(w.P, NP, nslots, lane, a0, a1, a2, k, tab); },
        m, it, ev, hist);
    if (lane == 0) {
        mp[0] = m[0]; mp[1] = m[1]; mp[2] = m[2];
        *fout = f;
        stats[0] = it; stats[1] = ev;
    }
}
template <int SLOTS>
__global__ void probe_guess_kernel(DeviceData dd, FrameDesc fd, double delay, int iters,
                                   uint64_t key_prefix, int mode, double* out, unsigned* n_exact) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int NP = SLOTS * 32;
    const int lane = threadIdx.x & 31;
    const WarpSmem w = warp_smem(smem_raw, 0, NP);
    const int nslots = (fd.n + 31) >> 5;
    build_rows_smem(dd, fd, delay, lane, w, NP);
    double M[3];
    if (mode == 2) {
        const Vec3 e = warp_ransac_exact<SLOTS>(dd, fd, w, iters, rng_task_key(key_prefix, fd.id), lane);
        M[0] = e.x; M[1] = e.y; M[2] = e.z;
    } else
        warp_ransac<SLOTS>(dd, fd, w, iters, rng_task_key(key_prefix, fd.id), lane, M, n_exact);
    __syncwarp();
    const double nrm = warp_norm_PM(w.P, NP, nslots, lane, M, nullptr);
    if (lane == 0) { out[0] = M[0]; out[1] = M[1]; out[2] = M[2]; out[3] = clamp_k(1.0 / nrm * 1e2); }
}

__global__ void fp64_peak_kernel(int iters, double* sink) {
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5,
           a6 = a0 + 6, a7 = a0 + 7;
    const double b = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
        a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
    }
    const double s = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (s == 12345.6789) sink[0] = s;
}

// ------------------------------------------------------------------------------------------
int slots_for(int max_n) {  // compile-time SLOTS instantiated for the estimator kernels
    const int need = (max_n + 31) / 32;
    const int have[] = {2, 4, 6, 7, 8, 12, 16};
    for (int v : have)
        if (need <= v) return v;
    return 16;
}

// Launch-configuration caches.  Both the opt-in to large dynamic shared memory
// (cudaFuncSetAttribute) and the occupancy of a kernel are properties of a (device, kernel) pair:
// a process may hold problems on several GPUs (rssync_create_multi), so everything here is keyed
// by the calling thread's current device.
int current_device() {
    int dev = 0;
    cudaGetDevice(&dev);
    return dev;
}
int sm_count_of(int dev) {
    static std::mutex mu;
    static std::map<int, int> cache;
    std::lock_guard<std::mutex> lk(mu);
    int& n = cache[dev];
    if (!n) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n;
}
// resident blocks per SM of `kernel` at this block size / shared memory size (>= 1); one occupancy
// query per (device, kernel, shared memory size): the Sync driver launches thousands of small
// kernels per second
template <class K>
int blocks_per_sm(K kernel, int threads, size_t smem) {
    static std::mutex mu;
    static std::map<std::tuple<int, const void*, size_t>, int> cache;
    std::lock_guard<std::mutex> lk(mu);
    int& slot = cache[std::make_tuple(current_device(), reinterpret_cast<const void*>(kernel), smem)];
    if (!slot) {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&slot, kernel, threads, smem);
        if (slot < 1) slot = 1;
    }
    return slot;
}
template <class K>
int grid_for(K kernel, size_t smem, long long warps_needed, int warps_per_block = kWarpsPerBlock) {
    const int per_sm = blocks_per_sm(kernel, warps_per_block * 32, smem);
    long long blocks_needed = (warps_needed + warps_per_block - 1) / warps_per_block;
    long long cap = (long long)sm_count_of(current_device()) * per_sm;
    long long g = blocks_needed < cap ? blocks_needed : cap;
    return (int)(g < 1 ? 1 : g);
}

template <class K>
void allow_smem(K kernel, size_t smem) {
    static std::mutex mu;
    static std::map<std::pair<int, const void*>, size_t> allowed;  // the largest size already granted
    std::lock_guard<std::mutex> lk(mu);
    size_t& have = allowed[{current_device(), reinterpret_cast<const void*>(kernel)}];
    if (smem <= have) return;
    cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    have = smem;
}

#define RS_DISPATCH_SLOTS(max_n, ...)                              \
    switch (slots_for(max_n)) {                                        \
        case 2: { constexpr int SL = 2; __VA_ARGS__; } break;          \
        case 4: { constexpr int SL = 4; __VA_ARGS__; } break;          \
        case 6: { constexpr int SL = 6; __VA_ARGS__; } break;          \
        case 7: { constexpr int SL = 7; __VA_ARGS__; } break;          \
        case 8: { constexpr int SL = 8; __VA_ARGS__; } break;          \
        case 12: { constexpr int SL = 12; __VA_ARGS__; } break;        \
        default: { constexpr int SL = 16; __VA_ARGS__; } break;        \
    }

}  // namespace

// RS_CHECKED builds: line of the first failed device-side assertion (0: none).  The slot is mapped
// host memory, one per device, registered with that device's copy of g_assert_slot on first use.
int checked_assert_line() {
#ifdef RS_CHECKED
    static std::mutex mu;
    static std::map<int, int*> slots;
    std::lock_guard<std::mutex> lk(mu);
    const int dev = current_device();
    int*& h = slots[dev];
    if (!h) {
        cudaHostAlloc((void**)&h, sizeof(int), cudaHostAllocMapped);
        *h = 0;
        int* d = nullptr;
        cudaHostGetDevicePointer((void**)&d, h, 0);
        cudaMemcpyToSymbol(g_assert_slot, &d, sizeof(d));
        return 0;
    }
    return *(volatile int*)h;
#else
    return 0;
#endif
}

uint64_t launch_count() { return g_launches.load(); }
void count_launches(uint64_t n) { g_launches += n; }

int presync_max_chunk(const double* h_delays, int D, double frame_span_s, double sample_rate, int max_n) {
    if (D <= 1) return 1;
    int recs = 0;
    RS_DISPATCH_SLOTS(max_n, { recs = GridCfg<SL>::kRecs; });
    // a chunk of c consecutive delays spans at most (c - 1) * max |step| seconds; its window holds
    // floor(x_hi) + 2 - (floor(x_lo) - 1) + 1 <= (span + range) * sr + 5 records (grid_stage_unit)
    double step = 0.0;
    for (int i = 1; i < D; ++i) step = std::max(step, std::fabs(h_delays[i] - h_delays[i - 1]));
    const double room = ((double)recs - 5.0) / sample_rate - frame_span_s;  // seconds of delay range
    if (!(room > 0.0) || !(step == step)) return 1;
    if (step <= 0.0) return D;
    const double c = std::floor(room / step) + 1.0;
    return (int)std::max(1.0, std::min(c, (double)D));
}

void launch_presync_tasks(const DeviceData& dd, const FrameDesc* d_frames, int F, int max_n,
                          const double* d_delays, int D, uint64_t seed, uint64_t stream, uint64_t call_no,
                          uint64_t idx_base, double* d_framecost, int cost_stride, unsigned* d_flags,
                          cudaStream_t st, const uint64_t* d_frame_call_no, int max_chunk, bool simplified,
                          int spare_sms) {
    if (F <= 0 || D <= 0) return;
    RS_DISPATCH_SLOTS(max_n, {
        using Cfg = GridCfg<SL>;
        auto kern = simplified ? presync_kernel<SL, true> : presync_kernel<SL, false>;
        allow_smem(kern, Cfg::kSmem);
        const int sm_count = sm_count_of(current_device());
        const int per_sm = blocks_per_sm(kern, Cfg::kWarps * 32, Cfg::kSmem);
        const long long blocks_cap = (long long)std::max(1, sm_count - std::max(0, spare_sms)) * per_sm;
        // Delays per unit: as many as the staged window takes (max_chunk; 0 = unknown, be conservative),
        // but no more than leaves every block several units (small grids: PreSync on a 60-frame window),
        // and at least one task per warp when the grid has that many delays.
        int chunk = std::min(D, max_chunk > 0 ? max_chunk : Cfg::kWarps * 2);
        const long long cpf_par = (blocks_cap * 4 + F - 1) / F;  // units per frame for 4 units per block
        const int chunk_par = (int)std::max<long long>(1, (D + cpf_par - 1) / cpf_par);
        chunk = std::min(chunk, std::max(chunk_par, std::min(D, Cfg::kWarps)));
        const int cpf = (D + chunk - 1) / chunk;
        chunk = (D + cpf - 1) / cpf;  // balanced
        const long long units = (long long)F * cpf;
        const int grid = (int)std::max<long long>(1, std::min<long long>(units, blocks_cap));
        const int staged = chunk >= Cfg::kWarps ? 1 : 0;
        kern<<<grid, Cfg::kWarps * 32, Cfg::kSmem, st>>>(dd, d_frames, F, d_delays, D, chunk, cpf, seed, stream,
                                                         call_no, d_frame_call_no, idx_base, d_framecost,
                                                         cost_stride, d_flags, staged);
    });
    g_launches += 1;
}

void launch_presync_reduce(const double* d_framecost, int F, int D, double* d_costs, cudaStream_t st,
                           const int* d_win_begin, int n_windows) {
    if (D <= 0) return;
    if (F <= 0) {
        cudaMemsetAsync(d_costs, 0, sizeof(double) * D * (d_win_begin ? n_windows : 1), st);
        return;
    }
    if (d_win_begin)
        reduce_windows_kernel<<<(n_windows * D + 3) / 4, 128, 0, st>>>(d_framecost, D, F, d_win_begin,
                                                                      n_windows, d_costs);
    else
        reduce_rows_kernel<<<(D + 3) / 4, 128, 0, st>>>(d_framecost, D, F, d_costs);
    g_launches += 1;
}

void launch_presync_grid(const DeviceData& dd, const FrameDesc* d_frames, int F, int max_n,
                         const double* d_delays, int D, uint64_t seed, uint64_t stream,
                         uint64_t call_no, uint64_t idx_base, double* d_framecost, double* d_costs,
                         unsigned* d_flags, cudaStream_t st, int max_chunk, bool simplified,
                         const uint64_t* d_frame_call_no, const int* d_win_begin, int n_windows) {
    launch_presync_tasks(dd, d_frames, F, max_n, d_delays, D, seed, stream, call_no, idx_base, d_framecost, F,
                         d_flags, st, d_frame_call_no, max_chunk, simplified);
    launch_presync_reduce(d_framecost, F, D, d_costs, st, d_win_begin, n_windows);
}

void launch_sync_init(const DeviceData& dd, const SyncBatchDev& b, const double* d_sp_delay,
                      const uint64_t* d_sp_callno, const unsigned char* d_sp_active, uint64_t seed,
                      cudaStream_t st) {
    if (b.T <= 0) return;
    RS_DISPATCH_SLOTS(b.max_n, {
        auto kern = sync_init_kernel<SL>;
        const size_t smem = (size_t)kWarpsPerBlock * warp_smem_bytes(SL * 32);
        allow_smem(kern, smem);
        const int grid = grid_for(kern, smem, b.T);
        kern<<<grid, kWarpsPerBlock * 32, smem, st>>>(dd, b, d_sp_delay, d_sp_callno, d_sp_active, seed);
    });
    g_launches += 1;
}

void launch_sync_motion_fgrad(const DeviceData& dd, const SyncBatchDev& b, const double* d_sp_delay,
                              const double* d_sp_x0, const unsigned char* d_sp_active,
                              double* d_task_scratch, double* d_out_v, double* d_out_g,
                              double* d_trial_delay, int ntrial, int* d_lbfgs_stats,
                              unsigned long long* d_evals_total, bool many_tasks, cudaStream_t st) {
    // A lane whose syncpoints hold no frames (T == 0) still needs its sums: the reference adds over
    // an empty frame list, cost 0 and gradient 0 (core_private.cpp:228-240), and the host's
    // Backtrack / momentum step reads them -- only the per-task kernel is skipped.
    if (b.S <= 0) return;
    auto launch = [&](auto kern, int W) {
        const size_t smem = kLog1pTableBytes + (size_t)W * warp_smem_bytes(slots_for(b.max_n) * 32) +
                            (size_t)W * kLbfgsHistDoubles * sizeof(double);
        allow_smem(kern, smem);
        const int grid = grid_for(kern, smem, b.T, W);
        kern<<<grid, W * 32, smem, st>>>(dd, b, d_sp_delay, d_sp_x0, d_sp_active, d_task_scratch, d_lbfgs_stats,
                                         d_evals_total);
    };
    if (b.T > 0) RS_DISPATCH_SLOTS(b.max_n, {
        if (many_tasks) launch(sync_motion_fgrad_kernel<SL, true>, LbfgsCfg<true>::kWarps);
        else launch(sync_motion_fgrad_kernel<SL, false>, LbfgsCfg<false>::kWarps);
    });
    reduce_fgrad_kernel<<<(b.S + 3) / 4, 128, 0, st>>>(b, d_sp_active, d_task_scratch, d_sp_x0, d_out_v,
                                                       d_out_g, d_trial_delay, ntrial);
    g_launches += 2;
}

void launch_sync_trials(const DeviceData& dd, const SyncBatchDev& b, const double* d_trial_delay,
                        int ntrial, const unsigned char* d_sp_active, double* d_task_scratch,
                        double* d_out, cudaStream_t st, const double* d_n_eval) {
    if (b.S <= 0 || ntrial <= 0) return;
    if (b.T > 0) {  // (T == 0: sums over no frames, see launch_sync_motion_fgrad)
        const int NP = slots_for(b.max_n) * 32;
        const size_t smem = kLog1pTableBytes + (size_t)kWarpsPerBlock * warp_smem_bytes(NP);
        allow_smem(sync_trials_kernel, smem);
        const int grid = grid_for(sync_trials_kernel, smem, (long long)b.T * ntrial);
        sync_trials_kernel<<<grid, kWarpsPerBlock * 32, smem, st>>>(dd, b, NP, d_trial_delay, ntrial,
                                                                    d_sp_active, d_task_scratch, d_n_eval);
    }
    reduce_trials_kernel<<<(b.S * ntrial + 3) / 4, 128, 0, st>>>(b, ntrial, d_sp_active, d_task_scratch, d_out,
                                                                 d_n_eval);
    g_launches += 2;
}

void launch_probe_problem_matrix(const DeviceData& dd, FrameDesc fd, double delay, double* d_P,
                                 cudaStream_t st) {
    const int NP = slots_for(fd.n) * 32;
    probe_problem_kernel<<<1, 32, warp_smem_bytes(NP), st>>>(dd, fd, NP, delay, d_P);
    g_launches += 1;
}
void launch_probe_log1p(const double* d_x, int n, double* d_out, cudaStream_t st) {
    probe_log1p_kernel<<<(n + 255) / 256, 256, 0, st>>>(d_x, n, d_out);
    g_launches += 1;
}
void launch_probe_loss(const DeviceData& dd, FrameDesc fd, double delay, const double* d_m, double k,
                       double* d_out, cudaStream_t st) {
    const int NP = slots_for(fd.n) * 32;
    probe_loss_kernel<<<1, 32, kLog1pTableBytes + warp_smem_bytes(NP), st>>>(dd, fd, NP, delay, d_m, k, d_out);
    g_launches += 1;
}
void launch_probe_lbfgs(const DeviceData& dd, FrameDesc fd, double delay, double* d_m, double k,
                        double* d_f, int* d_stats, cudaStream_t st) {
    const int NP = slots_for(fd.n) * 32;
    probe_lbfgs_kernel<<<1, 32, kLog1pTableBytes + warp_smem_bytes(NP), st>>>(dd, fd, NP, delay, d_m, k, d_f, d_stats);
    g_launches += 1;
}
void launch_probe_guess(const DeviceData& dd, FrameDesc fd, double delay, int iters,
                        uint64_t key_prefix, int mode, double* d_mk, unsigned* d_n_exact,
                        cudaStream_t st) {
    RS_DISPATCH_SLOTS(fd.n, {
        auto kern = probe_guess_kernel<SL>;
        kern<<<1, 32, warp_smem_bytes(SL * 32), st>>>(dd, fd, delay, iters, key_prefix, mode,
                                                            d_mk, d_n_exact);
    });
    g_launches += 1;
}

void launch_ingest_pixels(const PixelFrame* d_frames, int n_frames, const double* d_points_a,
                          const double* d_points_b, LensDev lens, double image_rows, double* d_rays,
                          int32_t* d_orig, int32_t* d_pos, double* d_rowq, cudaStream_t st) {
    if (n_frames <= 0) return;
    ingest_pixels_kernel<<<n_frames, kIngestThreads, 0, st>>>(d_frames, d_points_a, d_points_b, lens,
                                                               image_rows, d_rays, d_orig, d_pos,
                                                               reinterpret_cast<double2*>(d_rowq));
    g_launches += 1;
}

void launch_retime_frames(const PixelFrame* d_frames, int n_frames, const double* d_src_rays,
                          const int32_t* d_src_orig, const double* d_rowq, double readout, double* d_rays,
                          int32_t* d_orig, int32_t* d_pos, double* d_ext, cudaStream_t st) {
    if (n_frames <= 0) return;
    retime_frames_kernel<<<n_frames, kIngestThreads, 0, st>>>(d_frames, d_src_rays, d_src_orig,
                                                               reinterpret_cast<const double2*>(d_rowq), readout,
                                                               d_rays, d_orig, d_pos,
                                                               reinterpret_cast<double4*>(d_ext));
    g_launches += 1;
}

void launch_ingest_rays(const PixelFrame* d_frames, int n_frames, const double* d_ts_a,
                        const double* d_ts_b, const double* d_rays_a, const double* d_rays_b,
                        double* d_rays, int32_t* d_orig, int32_t* d_pos, cudaStream_t st) {
    if (n_frames <= 0) return;
    ingest_rays_kernel<false><<<n_frames, kIngestThreads, 0, st>>>(d_frames, d_ts_a, d_ts_b, d_rays_a, d_rays_b,
                                                                    0.0, d_rays, d_orig, d_pos, nullptr);
    g_launches += 1;
}

void launch_ingest_row_fractions(const PixelFrame* d_frames, int n_frames, const double* d_frac_a,
                                 const double* d_frac_b, const double* d_rays_a, const double* d_rays_b,
                                 double readout, double* d_rays, int32_t* d_orig, int32_t* d_pos, double* d_rowq,
                                 cudaStream_t st) {
    if (n_frames <= 0) return;
    ingest_rays_kernel<true><<<n_frames, kIngestThreads, 0, st>>>(d_frames, d_frac_a, d_frac_b, d_rays_a, d_rays_b,
                                                                   readout, d_rays, d_orig, d_pos,
                                                                   reinterpret_cast<double2*>(d_rowq));
    g_launches += 1;
}

void launch_stage_rays(const int64_t* d_at, int n_frames, int64_t total, const double* rays_a,
                       const double* rays_b, const double* ts_a, const double* ts_b, double* d_stage,
                       StageInfo* d_info, cudaStream_t st) {
    if (n_frames <= 0) return;
    // staged as ingest_rays_kernel reads it: ts_a, ts_b, rays_a, rays_b
    StageArgs a{d_at, total, {rays_a, rays_b, ts_a, ts_b},
                {d_stage + 2 * total, d_stage + 5 * total, d_stage, d_stage + total}, nullptr, 0.0, 1.0, d_info};
    stage_tracks_kernel<StageMode::kRays><<<n_frames, kStageThreads, 0, st>>>(a);
    g_launches += 1;
}

void launch_stage_row_fractions(const int64_t* d_at, const double* d_frame_ts, int n_frames, int64_t total,
                                const double* rays_a, const double* rays_b, const double* frac_a,
                                const double* frac_b, double readout, double* d_stage, StageInfo* d_info,
                                cudaStream_t st) {
    if (n_frames <= 0) return;
    // ingest_rays_kernel's layout with the fractions in the ts slots: frac_a, frac_b, rays_a, rays_b
    StageArgs a{d_at, total, {rays_a, rays_b, frac_a, frac_b},
                {d_stage + 2 * total, d_stage + 5 * total, d_stage, d_stage + total}, d_frame_ts, readout, 1.0,
                d_info};
    stage_tracks_kernel<StageMode::kRowFractions><<<n_frames, kStageThreads, 0, st>>>(a);
    g_launches += 1;
}

void launch_stage_points(const int64_t* d_at, const double* d_frame_ts, int n_frames, int64_t total,
                         const double* points_a, const double* points_b, const LensDev& lens, double rows,
                         double* d_stage, StageInfo* d_info, cudaStream_t st) {
    if (n_frames <= 0) return;
    StageArgs a{d_at, total, {points_a, points_b, nullptr, nullptr}, {d_stage, d_stage + 2 * total, nullptr, nullptr},
                d_frame_ts, lens.ro, rows, d_info, lens.fx, lens.fy, lens.cx, lens.cy};
    stage_tracks_kernel<StageMode::kPoints><<<n_frames, kStageThreads, 0, st>>>(a);
    g_launches += 1;
}

namespace {
TrackPyr track_pyr(const TrackImages& im, float* d_pyr, int slots) {
    TrackPyr P{};
    P.im = im;
    P.slots = slots;
    P.scale = std::ldexp(1.f, -im.shift);
    P.w[0] = im.w0;
    P.h[0] = im.h0;
    size_t at = 0;
    for (int l = 1; l < im.levels; ++l) {
        P.w[l] = (P.w[l - 1] + 1) / 2;
        P.h[l] = (P.h[l - 1] + 1) / 2;
        P.lvl[l] = d_pyr + at;
        at += (size_t)slots * P.w[l] * P.h[l];
    }
    return P;
}
}  // namespace

size_t track_pyramid_floats(int w0, int h0, int levels) {
    size_t n = 0;
    for (int l = 1, w = w0, h = h0; l < levels; ++l) {
        w = (w + 1) / 2;
        h = (h + 1) / 2;
        n += (size_t)w * h;
    }
    return n;
}

size_t track_select_smem(int cell, int block, int sample) {
    const int r = block / 2, PW = cell + 2 * (r + 2), SW = cell + 2, GW = SW + 2 * r, GR = kSelStrip + 2 * r;
    return ((size_t)SW * SW + 2 * (size_t)GR * GW + 3 * (size_t)GR * SW) * sizeof(float) + (size_t)PW * PW * sample;
}

namespace {
template <typename T>
void launch_track_frames_t(const TrackImages& im, int n_frames, const int64_t* h_q_at, int64_t* d_q_at,
                           double* d_points, float* d_pyr, int slots, double* d_tracked, uint8_t* d_status,
                           unsigned* d_flag, const TrackExtra& ex, cudaStream_t st) {
    const TrackPyr P = track_pyr(im, d_pyr, slots);
    const int pw = im.window + 2;
    const size_t smem = (size_t)kLkWarps * (pw * pw + 2 * im.window * im.window) * sizeof(float);
    const TrackMask* M = ex.mask;
    if (M) allow_smem(track_lk_kernel<T, false, true>, smem);
    else allow_smem(track_lk_kernel<T, false>, smem);
    const bool back = ex.fb_max > 0.0;
    if (back) allow_smem(track_lk_kernel<T, true>, smem);
    const TrackSelect* S = ex.sel;
    const size_t sel_smem = S ? track_select_smem(S->cell, S->block, (int)sizeof(T)) : 0;
    if (S && M) allow_smem(select_cells_kernel<T, true>, sel_smem);
    else if (S) allow_smem(select_cells_kernel<T>, sel_smem);
    // a shared mask is eroded once, per-image masks with their pyramids
    const bool per_image = M && M->image_stride != 0;
    const TrackElig E{M ? M->d_elig : nullptr, per_image ? (int64_t)im.w0 * im.h0 : 0, per_image ? slots : 1};
    auto erode = [&](int j0, int n) {
        const dim3 grid((im.w0 + kErTX - 1) / kErTX, (im.h0 + kErTY - 1) / kErTY, n);
        track_erode_kernel<<<grid, 256, 0, st>>>(*M, im.w0, im.h0, j0, E);
        g_launches += 1;
    };
    if (M && !per_image) erode(0, 1);
    // chunk: build the pyramids of images [built, e), then track frames [f0, e - 1); image f0 is the
    // last one of the previous chunk, still in its slot
    for (int f0 = 0, built = 0; f0 < n_frames;) {
        const int e = std::min(n_frames + 1, f0 + slots);
        for (int l = 0; l + 1 < im.levels && e > built; ++l) {
            const dim3 grid((P.w[l + 1] + kPyrTX - 1) / kPyrTX, (P.h[l + 1] + kPyrTY - 1) / kPyrTY, e - built);
            track_pyramid_kernel<T><<<grid, kPyrTX * kPyrTY, 0, st>>>(P, l, built);
            g_launches += 1;
        }
        if (per_image && e > built) erode(built, e - built);
        // selection on the chunk's side-a images f0 .. e - 2; the tracker's grid then covers the bound
        // max_points per frame and its warps past q_at[e - 1] return at once
        const int nf = e - 1 - f0;
        if (S) {
            const dim3 grid(S->cells_x * S->cells_y, nf);
            if (M) select_cells_kernel<T, true><<<grid, kSelThreads, sel_smem, st>>>(im, *S, f0, E);
            else select_cells_kernel<T><<<grid, kSelThreads, sel_smem, st>>>(im, *S, f0, E);
            select_points_kernel<<<nf, kPickThreads, 0, st>>>(*S);
            select_prefix_kernel<<<1, kPickThreads, 0, st>>>(*S, d_q_at, f0, e - 1, im.w0, d_points);
            g_launches += 3;
        }
        const int64_t pts = S ? (int64_t)nf * S->max_points : h_q_at[e - 1] - h_q_at[f0];
        if (pts > 0) {
            const unsigned blocks = (unsigned)((pts + kLkWarps - 1) / kLkWarps);
            if (M)
                track_lk_kernel<T, false, true><<<blocks, kLkWarps * 32, smem, st>>>(
                    P, d_q_at, f0, e - 1, d_points, d_tracked, d_status, d_flag, 0.0, nullptr, E);
            else
                track_lk_kernel<T, false><<<blocks, kLkWarps * 32, smem, st>>>(P, d_q_at, f0, e - 1, d_points,
                                                                              d_tracked, d_status, d_flag, 0.0,
                                                                              nullptr, E);
            g_launches += 1;
            if (back) {
                track_lk_kernel<T, true><<<blocks, kLkWarps * 32, smem, st>>>(P, d_q_at, f0, e - 1, d_points,
                                                                             d_tracked, d_status, d_flag, ex.fb_max,
                                                                             ex.d_fb, E);
                g_launches += 1;
            }
        }
        built = e;
        f0 = e - 1;
    }
}
}  // namespace

void launch_track_frames(const TrackImages& im, int n_frames, const int64_t* h_q_at, int64_t* d_q_at,
                         double* d_points, float* d_pyr, int slots, double* d_tracked, uint8_t* d_status,
                         unsigned* d_flag, const TrackExtra& ex, cudaStream_t st) {
    if (n_frames <= 0) return;
    if (im.sample == 2)
        launch_track_frames_t<uint16_t>(im, n_frames, h_q_at, d_q_at, d_points, d_pyr, slots, d_tracked, d_status,
                                        d_flag, ex, st);
    else
        launch_track_frames_t<uint8_t>(im, n_frames, h_q_at, d_q_at, d_points, d_pyr, slots, d_tracked, d_status,
                                       d_flag, ex, st);
}

void launch_track_compact(const int64_t* d_q_at, int n_frames, const double* d_points, const double* d_tracked,
                          const uint8_t* d_status, double* d_out_a, double* d_out_b, int64_t* d_kept_at,
                          cudaStream_t st) {
    if (n_frames <= 0) return;
    track_compact_kernel<<<1, kCompactThreads, 0, st>>>(d_q_at, n_frames, d_points, d_tracked, d_status, d_out_a,
                                                        d_out_b, d_kept_at);
    g_launches += 1;
}

void launch_spline_finish(const double* d_quats, const double* d_rhs, const double* d_diag, int n,
                          double* d_rec, cudaStream_t st) {
    if (n <= 0) return;
    const long long threads = 4LL * n;
    spline_finish_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(d_quats, d_rhs, d_diag, n, d_rec);
    g_launches += 1;
}

void launch_gyro_integrate(const double* d_ts, const double* d_gyro, int n, const double* h_matrices, int n_var,
                           void* d_orients, double* d_quats, double* d_prefix, cudaStream_t st) {
    if (n <= 0 || n_var <= 0) return;
    static_assert(sizeof(OrientDev) == 9 * sizeof(double), "OrientDev is one 3x3 matrix");
    cudaMemcpyAsync(d_orients, h_matrices, sizeof(OrientDev) * (size_t)n_var, cudaMemcpyHostToDevice, st);  // pageable: staged before return
    const int nb = (n + (int)kGyroScanBlock - 1) / (int)kGyroScanBlock;
    gyro_local_kernel<<<(nb * n_var + 31) / 32, 32, 0, st>>>(d_ts, d_gyro, n, static_cast<const OrientDev*>(d_orients), n_var, d_quats);
    gyro_prefix_kernel<<<(n_var + 31) / 32, 32, 0, st>>>(d_quats, n, n_var, d_prefix);
    const long long total = (long long)n * n_var;
    gyro_apply_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_prefix, n, n_var, d_quats);
    g_launches += 3;
}
size_t gyro_orient_bytes(int n_var) { return sizeof(OrientDev) * (size_t)n_var; }
size_t gyro_prefix_doubles(int n, int n_var) {
    return (size_t)n_var * ((size_t)(n + (int)kGyroScanBlock - 1) / kGyroScanBlock + 1) * 4;
}

void launch_gyro_resample(const int64_t* d_ts_us, int count, const double* d_quats, int n_var, uint64_t tick0,
                          unsigned rate_hz, int n_out, double* d_out, unsigned* d_nonfinite, cudaStream_t st) {
    if (n_out <= 0 || n_var <= 0) return;
    const long long total = (long long)n_out * n_var;
    resample_kernel<<<(unsigned)((total + 127) / 128), 128, 0, st>>>(d_ts_us, count, d_quats, n_var, tick0, rate_hz, n_out,
                                                                     d_out, d_nonfinite);
    g_launches += 1;
}

void launch_spline_chains(const double* d_y, const double* d_f_down, const double* d_f_up, int n, int n_var,
                          double* d_rhs, cudaStream_t st) {
    if (n < 2 || n_var <= 0) return;
    spline_chains_kernel<<<(4 * n_var + 31) / 32, 32, 0, st>>>(d_y, d_f_down, d_f_up, n, n_var, d_rhs);
    g_launches += 1;
}

void launch_probe_trig(const double* d_x, int n, int which, double* d_out, cudaStream_t st) {
    probe_trig_kernel<<<(n + 255) / 256, 256, 0, st>>>(d_x, n, which, d_out);
    g_launches += 1;
}

float run_fp64_peak(int blocks, int threads, int iters, double* d_sink, cudaStream_t st) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    fp64_peak_kernel<<<blocks, threads, 0, st>>>(iters / 8 + 1, d_sink);  // warm-up
    cudaEventRecord(e0, st);
    fp64_peak_kernel<<<blocks, threads, 0, st>>>(iters, d_sink);
    cudaEventRecord(e1, st);
    cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    g_launches += 2;
    return ms;
}

}  // namespace rs
