// ORACLE — TEST INFRASTRUCTURE ONLY (see oracle/README.md).  CPU restatement of the rs-sync
// synchronisation loss engine: everything behind ISyncProblem (src/core/public/rssync.h:9-31 of
// the reference), i.e. src/core/core_private.cpp plus the src/core_support helpers it calls.
// Each function cites the reference lines it follows.  Exposed through a plain C interface so
// tests can drive it with ctypes.  Not linked into, loaded by, or called from the product.
//
// Parity status: the reference ships no golden vectors or tests (SURVEY.md §4).  This
// restatement is pinned against (a) analytic / SciPy known answers (tests/test_oracle_*.py) and
// (b) the UNMODIFIED reference translation units compiled here against a small Armadillo /
// ensmallen shim (oracle/_ref, built by oracle/Makefile) with the same pinned RNG.  Two pieces
// remain unpinned by construction and are stated as such in DESIGN.md: the RNG itself (the
// reference seeds mt19937 from random_device) and ens::L_BFGS (un-vendored third-party code,
// restated from its published algorithm).
#include "oracle_math.hpp"
#include "spec_trig.hpp"
#include "oracle_strict.hpp"

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <string>
#include <thread>
#include <vector>

using namespace orc;

namespace {

struct Frame {
    int n = 0;
    std::vector<double> ts_a, ts_b, ra, rb;  // ra/rb: xyz interleaved, 3*n
    std::vector<int> order;  // ray indices sorted by (ts_a, index): the spec's summation order
};

// Sums over the rays of one frame (the spec; stands in for arma::accu / arma::sum / arma::norm's
// inner sum, core_private.cpp:79,85,122; inline_utils.hpp:32-36, whose order is Armadillo's
// business).  The rays are visited in the order (ts_a, caller index); ray j of that order is added
// to partial sum j % 32, and the 32 partial sums are combined by an xor butterfly (strides 16, 8,
// 4, 2, 1).  A fixed order, so the value is reproducible bit for bit -- it is the order in which a
// warp whose lane l owns rays l, l + 32, ... adds them up.
struct RaySum {
    double lane[32];
    RaySum() { for (double& x : lane) x = 0.0; }
    inline void add(int j, double x) { lane[j & 31] += x; }
    double value() const {
        double a[32], b[32];
        for (int l = 0; l < 32; ++l) a[l] = lane[l];
        for (int off = 16; off >= 1; off >>= 1) {
            for (int l = 0; l < 32; ++l) b[l] = a[l] + a[l ^ off];
            for (int l = 0; l < 32; ++l) a[l] = b[l];
        }
        return a[0];
    }
};

struct Oracle {
    // gyro spline: OptData::quats / quats_start / sample_rate (core_private.hpp:15-22)
    double q0 = 0.0, sr = 0.0;
    long nq = 0;
    std::vector<double> rec;  // nq * 16
    std::vector<double> resampled;  // last resampled quaternions (4*nq) for tests
    std::map<int64_t, Frame> frames;
    uint64_t seed = 100, call_no = 0;
    int threads = 1;
    std::string err;
    // strict mode (oracle_strict.hpp): the reference's own expression order, plain sums, libm
    // log1p, and frames visited in `frame_order` (the reference's unordered_map order) — used to
    // compare control flow with the compiled reference bit for bit
    bool strict = false;
    std::vector<int64_t> frame_order;
    // simplified (no-translation) loss mode, thesis pdf-p.27-28 section 2.11 (no code in the reference
    // checkout): the residual of a ray pair is |ar x br| itself -- the de-rotated rays of a purely
    // rotating camera coincide -- instead of its component along the translation direction; no
    // estimator, no per-frame L-BFGS.  Definition shared with the engine (include/rssync_b200.h).
    bool simplified = false;
};

enum { OK = 0, E_INVALID = 1, E_NONFINITE = 2, E_ORDER = 3, E_STATE = 4 };

bool all_finite(const double* p, size_t n) {
    for (size_t i = 0; i < n; ++i)
        if (!std::isfinite(p[i])) return false;
    return true;
}

// ndspline::make (ndspline.cpp:13-19): one scalar spline per quaternion component.
void build_spline(Oracle& o, const double* quats, long n) {
    o.nq = n;
    o.rec.assign((size_t)n * 16, 0.0);
    for (int c = 0; c < 4; ++c) spline_build_1d(quats + c, n, 4, o.rec.data(), c);
}

// quat_slerp (quat.cpp:55-74).  4-term dot accumulated left to right.  spec: the contract's acos / sin
// (spec_trig.hpp), what the engine computes; otherwise libm, what the reference calls.
void slerp(const double p[4], const double qin[4], double t, double out[4], bool spec = false) {
    double q[4] = {qin[0], qin[1], qin[2], qin[3]};
    double d = ((p[0] * q[0] + p[1] * q[1]) + p[2] * q[2]) + p[3] * q[3];
    if (d < 0) {
        for (int i = 0; i < 4; ++i) q[i] = -q[i];
        d = ((p[0] * q[0] + p[1] * q[1]) + p[2] * q[2]) + p[3] * q[3];
    }
    double m1, m2;
    const double theta = spec ? orc::spec_acos(d) : std::acos(d);
    if (theta > 1e-9) {
        const double st = spec ? orc::spec_sin(theta) : std::sin(theta);
        m1 = (spec ? orc::spec_sin((1 - t) * theta) : std::sin((1 - t) * theta)) / st;
        m2 = (spec ? orc::spec_sin(t * theta) : std::sin(t * theta)) / st;
    } else {
        m1 = 1 - t;
        m2 = t;
    }
    for (int i = 0; i < 4; ++i) out[i] = m1 * p[i] + m2 * q[i];
}

// opt_compute_problem (core_private.cpp:15-32)
void problem_matrix(const Oracle& o, const Frame& f, double delay, double* P) {
    if (o.strict) {
        for (int i = 0; i < f.n; ++i)
            orc_strict::problem_row(o.rec.data(), o.nq, o.q0, o.sr, delay, f.ts_a[i], f.ts_b[i],
                                    &f.ra[3 * i], &f.rb[3 * i], P + 3 * i);
        return;
    }
    for (int i = 0; i < f.n; ++i)
        problem_row(o.rec.data(), o.nq, o.q0, o.sr, delay, f.ts_a[i], f.ts_b[i], &f.ra[3 * i],
                    &f.rb[3 * i], P + 3 * i);
}

// opt_guess_translational_motion (core_private.cpp:34-59) with the pinned RNG.
void guess_motion(const double* P, int n, int iters, uint64_t key, double best[3],
                  std::vector<double>& nP, std::vector<double>& r2, bool strict = false) {
    nP.resize((size_t)n * 3);
    r2.resize(n);
    if (strict) {
        for (int i = 0; i < n; ++i) orc_strict::safe_normalize3(P + 3 * i, &nP[3 * i]);
        double least = std::numeric_limits<double>::infinity();
        best[0] = best[1] = best[2] = 0.0;
        for (int it = 0; it < iters; ++it) {
            uint32_t a = rng_index(key, it, 0, n);
            uint32_t b, k = 1;
            do { b = rng_index(key, it, k++, n); } while (b == a);
            double c[3], v[3];
            orc_strict::cross3(P + 3 * a, P + 3 * b, c);
            orc_strict::safe_normalize3(c, v);
            for (int i = 0; i < n; ++i) {
                double r = orc_strict::dot3(&nP[3 * i], v);
                r2[i] = r * r;
            }
            std::nth_element(r2.begin(), r2.begin() + n / 4, r2.end());
            double med = r2[n / 4];
            if (med < least) { least = med; best[0] = v[0]; best[1] = v[1]; best[2] = v[2]; }
        }
        return;
    }
    for (int i = 0; i < n; ++i) safe_normalize3(P + 3 * i, &nP[3 * i]);  // :35-36
    double least = std::numeric_limits<double>::infinity();
    best[0] = best[1] = best[2] = 0.0;
    for (int it = 0; it < iters; ++it) {
        uint32_t a = rng_index(key, it, 0, n);  // :42
        uint32_t b, k = 1;
        do { b = rng_index(key, it, k++, n); } while (b == a);  // :43
        const double* pa = P + 3 * a;
        const double* pb = P + 3 * b;
        double c[3] = {hyp_cross_term(pa[1], pb[2], pa[2] * pb[1]), hyp_cross_term(pa[2], pb[0], pa[0] * pb[2]),
                       hyp_cross_term(pa[0], pb[1], pa[1] * pb[0])};
        double v[3];
        safe_normalize3(c, v);  // :45-46
        for (int i = 0; i < n; ++i) {
            double r = dot3(&nP[3 * i], v);  // :48
            r2[i] = r * r;                    // :49
        }
        std::nth_element(r2.begin(), r2.begin() + n / 4, r2.end());  // :51-52 (value at sorted[n/4])
        double med = r2[n / 4];
        if (med < least) {  // :53-56
            least = med;
            best[0] = v[0]; best[1] = v[1]; best[2] = v[2];
        }
    }
}

double norm_PM(const double* P, int n, const int* order, const double m[3]) {  // arma::norm(P * M)
    RaySum ss;
    for (int j = 0; j < n; ++j) {
        double pm = dot3(P + 3 * order[j], m);
        ss.add(j, pm * pm);
    }
    return std::sqrt(ss.value());
}

// simplified mode: the residual vector is the row norms; its 2-norm (the analogue of arma::norm(P * M))
double norm_rows(const double* P, int n, const int* order) {
    RaySum ss;
    for (int j = 0; j < n; ++j) {
        const double* r = P + 3 * order[j];
        const double nr = std::sqrt(dot3(r, r));
        ss.add(j, nr * nr);
    }
    return std::sqrt(ss.value());
}
// sum_i log1p((|P_i| k)^2)
double loss_rows_P(const double* P, int n, const int* order, double k) {
    RaySum acc;
    for (int j = 0; j < n; ++j) {
        const double* r = P + 3 * order[j];
        const double v = std::sqrt(dot3(r, r)) * k;
        acc.add(j, log1p_nonneg(v * v));
    }
    return acc.value();
}

// per-frame body of pre_sync (core_private.cpp:75-85) / DebugPreSync (:350-356)
double presync_frame_cost(const Oracle& o, const Frame& f, double delay, uint64_t key, int* flags) {
    std::vector<double> P((size_t)f.n * 3), nP, r2;
    problem_matrix(o, f, delay, P.data());
    if (flags && !all_finite(P.data(), P.size())) *flags |= 1;
    if (o.simplified) {  // same aggregation as :79-85 with the row norms as residuals
        const double k = clamp_k(1.0 / norm_rows(P.data(), f.n, f.order.data()) * 1e2);
        RaySum acc;
        for (int j = 0; j < f.n; ++j) {
            const double* row = &P[3 * f.order[j]];
            const double r = std::sqrt(dot3(row, row)) * k;
            if (flags && !std::isfinite(r)) *flags |= 4;
            const double rho = log1p_nonneg(r * r);
            if (flags && !std::isfinite(rho)) *flags |= 8;
            acc.add(j, std::sqrt(rho));
        }
        return std::sqrt(acc.value());
    }
    double M[3];
    guess_motion(P.data(), f.n, 20, key, M, nP, r2, o.strict);
    if (flags && !all_finite(M, 3)) *flags |= 2;
    if (o.strict) {
        double k = clamp_k(1 / orc_strict::norm_PM(P.data(), f.n, M) * 1e2);
        double scale = k / orc_strict::norm_seq(M, 3);
        double acc = 0.0;
        for (int i = 0; i < f.n; ++i) {
            double r = orc_strict::dot3(&P[3 * i], M) * scale;
            acc += std::sqrt(std::log1p(r * r));
        }
        return std::sqrt(acc);
    }
    double k = clamp_k(1.0 / norm_PM(P.data(), f.n, f.order.data(), M) * 1e2);  // :79
    double scale = k / std::sqrt(dot3(M, M));                                      // :80
    RaySum acc;
    for (int j = 0; j < f.n; ++j) {
        double r = dot3(&P[3 * f.order[j]], M) * scale;
        if (flags && !std::isfinite(r)) *flags |= 4;
        double rho = log1p_nonneg(r * r);  // :82
        if (flags && !std::isfinite(rho)) *flags |= 8;
        acc.add(j, std::sqrt(rho));
    }
    return std::sqrt(acc.value());  // :85
}

std::vector<const std::pair<const int64_t, Frame>*> select_frames(const Oracle& o, int64_t fb,
                                                                  int64_t fe_exclusive) {
    std::vector<const std::pair<const int64_t, Frame>*> v;
    if (!o.frame_order.empty()) {  // strict mode: the reference's unordered_map order
        for (int64_t id : o.frame_order) {
            auto it = o.frames.find(id);
            if (it != o.frames.end() && id >= fb && id < fe_exclusive) v.push_back(&*it);
        }
        return v;
    }
    for (auto& kv : o.frames)
        if (kv.first >= fb && kv.first < fe_exclusive) v.push_back(&kv);
    return v;
}

template <class F>
void parallel_for(int threads, size_t n, F&& fn) {
    if (threads <= 1 || n < 2) {
        for (size_t i = 0; i < n; ++i) fn(i);
        return;
    }
    std::atomic<size_t> next{0};
    std::vector<std::thread> pool;
    auto work = [&]() {
        for (;;) {
            size_t i = next.fetch_add(1);
            if (i >= n) break;
            fn(i);
        }
    };
    for (int t = 0; t < threads; ++t) pool.emplace_back(work);
    for (auto& t : pool) t.join();
}

// cost of every delay in `delays` over frames [fb, fe): the body of pre_sync's outer loop
// (core_private.cpp:69-88).  frame_costs (optional) receives n_delays x n_frames values.
int presync_grid(Oracle& o, int64_t fb, int64_t fe, const double* delays, int nd, uint64_t stream,
                 uint64_t call_no, uint64_t idx_base, double* costs, double* frame_costs,
                 int* flags_out) {
    if (o.nq < 2) { o.err = "gyro quaternions not set"; return E_STATE; }
    auto fr = select_frames(o, fb, fe);
    for (auto* kv : fr)
        if (kv->second.n < 2) { o.err = "frame with fewer than 2 rays"; return E_INVALID; }
    size_t nf = fr.size();
    std::vector<double> fc((size_t)nd * nf);
    std::vector<int> fl((size_t)nd * nf, 0);
    parallel_for(o.threads, (size_t)nd * nf, [&](size_t t) {
        size_t d = t / nf, j = t % nf;
        uint64_t key = rng_task_key(o.seed, stream, call_no, idx_base + d, fr[j]->first);
        fc[t] = presync_frame_cost(o, fr[j]->second, delays[d], key, &fl[t]);
    });
    int flags = 0;
    for (int d = 0; d < nd; ++d) {
        DD acc;
        double plain = 0.0;
        for (size_t j = 0; j < nf; ++j) {
            acc.add(fc[d * nf + j]);
            plain += fc[d * nf + j];
            flags |= fl[d * nf + j];
        }
        costs[d] = o.strict ? plain : acc.value();
    }
    if (frame_costs) std::copy(fc.begin(), fc.end(), frame_costs);
    if (flags_out) *flags_out = flags;
    return OK;
}

// ---------------------------------------------------------------------------------------------
// FrameState (core_private.hpp:24-42)
struct FrameState {
    const Frame* f;
    int64_t id;
    double m[3];
    double k = 1e3;
};

// FrameState::Loss, 3-argument form (core_private.cpp:117-123), on a prebuilt P.
double loss3_P(const double* P, int n, const int* order, const double m[3], double k) {
    double scale = k / std::sqrt(dot3(m, m));
    RaySum acc;
    for (int j = 0; j < n; ++j) {
        double r = dot3(P + 3 * order[j], m) * scale;
        acc.add(j, log1p_nonneg(r * r));
    }
    return acc.value();
}
double loss3(const Oracle& o, const Frame& f, double delay, const double m[3], double k) {
    std::vector<double> P((size_t)f.n * 3);
    problem_matrix(o, f, delay, P.data());
    if (o.simplified) return loss_rows_P(P.data(), f.n, f.order.data(), k);
    return o.strict ? orc_strict::loss3_P(P.data(), f.n, m, k) : loss3_P(P.data(), f.n, f.order.data(), m, k);
}

// FrameState::Loss, 5-argument form (core_private.cpp:92-115): value and d/dm in closed form
// of the forward-mode chain (inline_utils.hpp:19-48):
//   v1 = P m, den = |m|^2 / k^2, u_i = v1_i^2 / den, loss = sum log1p(u_i)
//   grad = sum_i 1/(1+u_i) * ( (2 v1_i / den) P_i - (v1_i^2 / den^2) (1/k^2) (2 m) )
double loss5_P(const double* P, int n, const int* order, const double m[3], double k, double grad[3]) {
    const double kk = k * k;
    const double den = dot3(m, m) / kk;
    const double inv_den = 1.0 / den;
    RaySum L, g0, g1, g2, su;
    for (int j = 0; j < n; ++j) {
        const double* p = P + 3 * order[j];
        double v1 = dot3(p, m);
        double u = (v1 * v1) * inv_den;
        L.add(j, log1p_nonneg(u));
        double w = 1.0 / (1.0 + u);
        double wv = w * v1;
        g0.add(j, wv * p[0]);
        g1.add(j, wv * p[1]);
        g2.add(j, wv * p[2]);
        su.add(j, w * u);
    }
    const double c1 = 2.0 * inv_den;
    const double c2 = (c1 / kk) * su.value();
    grad[0] = c1 * g0.value() - c2 * m[0];
    grad[1] = c1 * g1.value() - c2 * m[1];
    grad[2] = c1 * g2.value() - c2 * m[2];
    return L.value();
}

// ens::L_BFGS (ensmallen 2.x, un-vendored: vcpkg.json:8; call site core_private.cpp:264-294)
// restated from its published algorithm with the defaults numBasis=10, armijoConstant=1e-4,
// wolfe=0.9, factr=1e-15, maxLineSearchTrials=50, minStep=1e-20, maxStep=1e20 and the two
// overrides maxIterations=200, minGradientNorm=1e-4 (:265-266).  PARITY UNPINNED for this
// function: ensmallen is not available to check against.
struct LbfgsStats { int iters = 0, evals = 0; };
struct DotSpec { double operator()(const double* a, const double* b) const { return orc::dot3(a, b); } };
struct DotStrict { double operator()(const double* a, const double* b) const { return orc_strict::dot3(a, b); } };
template <class FG, class DOT = DotSpec>
double lbfgs3(FG&& fg, double x[3], LbfgsStats* st, DOT dot3 = DOT()) {
    const int numBasis = 10, maxIterations = 200, maxTrials = 50;
    const double minGradientNorm = 1e-4, armijo = 1e-4, wolfe = 0.9, factr = 1e-15,
                 minStep = 1e-20, maxStep = 1e20;
    double S[numBasis][3], Y[numBasis][3];
    double g[3], oldx[3], oldg[3], dir[3], trial[3];
    double f = fg(x, g);
    if (st) st->evals++;
    for (int it = 0; it != maxIterations; ++it) {
        double prevf = f;
        if (it > 0 && std::sqrt(dot3(g, g)) < minGradientNorm) break;
        if (std::isnan(f)) break;
        // scaling factor
        double scaling;
        if (it > 0) {
            int pp = (it - 1) % numBasis;
            double yy = dot3(Y[pp], Y[pp]);
            double denom = (yy >= 1e-10) ? yy : 1.0;
            scaling = dot3(S[pp], Y[pp]) / denom;
        } else {
            double gn = std::sqrt(dot3(g, g));
            scaling = (gn >= 1e-5) ? 1.0 / gn : 1.0;
        }
        if (scaling == 0.0 || !std::isfinite(scaling)) break;
        // two-loop recursion
        double rho[numBasis], alpha[numBasis];
        dir[0] = g[0]; dir[1] = g[1]; dir[2] = g[2];
        int limit = (numBasis > it) ? 0 : (it - numBasis);
        for (int i = it; i != limit; --i) {
            int tp = (i + (numBasis - 1)) % numBasis;
            double ys = dot3(Y[tp], S[tp]);
            rho[it - i] = (ys != 0) ? (1.0 / ys) : 1.0;
            alpha[it - i] = rho[it - i] * dot3(S[tp], dir);
            for (int c = 0; c < 3; ++c) dir[c] -= alpha[it - i] * Y[tp][c];
        }
        for (int c = 0; c < 3; ++c) dir[c] *= scaling;
        for (int i = limit; i < it; ++i) {
            int tp = i % numBasis;
            double beta = rho[it - i - 1] * dot3(Y[tp], dir);
            double coef = alpha[it - i - 1] - beta;
            for (int c = 0; c < 3; ++c) dir[c] += coef * S[tp][c];
        }
        for (int c = 0; c < 3; ++c) dir[c] = -dir[c];
        for (int c = 0; c < 3; ++c) { oldx[c] = x[c]; oldg[c] = g[c]; }
        // line search
        double step = 1.0, bestStep = 1.0, bestObj = std::numeric_limits<double>::max();
        const double init_dg = dot3(g, dir);
        if (init_dg > 0.0) break;  // not a descent direction: line search reports failure
        const double f0 = f;
        const double lin = armijo * init_dg;
        int trials = 0;
        for (;;) {
            for (int c = 0; c < 3; ++c) trial[c] = x[c] + step * dir[c];
            f = fg(trial, g);
            if (st) st->evals++;
            if (f < bestObj) { bestStep = step; bestObj = f; }
            trials++;
            double width;
            if (f > f0 + step * lin) {
                width = 0.5;
            } else {
                double dg = dot3(g, dir);
                if (dg < wolfe * init_dg) {
                    width = 2.1;
                } else if (dg > -wolfe * init_dg) {
                    width = 0.5;
                } else {
                    break;
                }
            }
            if (step < minStep || step > maxStep || trials >= maxTrials) break;
            step *= width;
        }
        for (int c = 0; c < 3; ++c) x[c] += bestStep * dir[c];
        if (st) st->iters++;
        if (bestStep == 0.0) break;
        double denom = std::max(std::max(std::fabs(prevf), std::fabs(f)), 1.0);
        if ((prevf - f) / denom <= factr) break;
        int op = it % numBasis;
        for (int c = 0; c < 3; ++c) { S[op][c] = x[c] - oldx[c]; Y[op][c] = g[c] - oldg[c]; }
    }
    return f;
}

struct SyncTrace { double* delays; double* steps; int cap; int n; };

// SyncProblemPrivate::Sync (core_private.cpp:211-334)
int sync_impl(Oracle& o, double initial_delay, int64_t fb, int64_t fe, double center, double radius,
              uint64_t call_no, double* out_cost, double* out_delay, SyncTrace* trace,
              long* counters) {
    if (o.nq < 2) { o.err = "gyro quaternions not set"; return E_STATE; }
    double delay = initial_delay;
    std::vector<FrameState> fs;
    std::vector<int64_t> order;
    if (!o.frame_order.empty()) order = o.frame_order;
    else for (auto& kv : o.frames) order.push_back(kv.first);
    for (int64_t id : order) {  // :218-223, inclusive frame_end
        auto itf = o.frames.find(id);
        if (itf == o.frames.end() || id < fb || id > fe) continue;
        if (itf->second.n < 2) { o.err = "frame with fewer than 2 rays"; return E_INVALID; }
        FrameState s;
        s.f = &itf->second;
        s.id = id;
        fs.push_back(s);
    }
    const bool strict = o.strict;
    long n_build = 0, n_lbfgs_eval = 0, n_lbfgs_iter = 0, n_outer = 0;
    parallel_for(o.threads, fs.size(), [&](size_t j) {  // GuessMotion + GuessK, :125-133
        FrameState& s = fs[j];
        std::vector<double> P((size_t)s.f->n * 3), nP, r2;
        problem_matrix(o, *s.f, delay, P.data());
        if (o.simplified) {  // no translation direction: only the scale k, from the row norms
            s.m[0] = s.m[1] = s.m[2] = 0.0;
            s.k = clamp_k(1.0 / norm_rows(P.data(), s.f->n, s.f->order.data()) * 1e2);
            return;
        }
        uint64_t key = rng_task_key(o.seed, kStreamSyncInit, call_no, 0, s.id);
        guess_motion(P.data(), s.f->n, 200, key, s.m, nP, r2, strict);
        s.k = strict ? clamp_k(1 / orc_strict::norm_PM(P.data(), s.f->n, s.m) * 1e2)
                     : clamp_k(1.0 / norm_PM(P.data(), s.f->n, s.f->order.data(), s.m) * 1e2);
    });
    n_build += (long)fs.size();

    auto sum_loss3 = [&](double x) {  // simple_objective, :242-252
        std::vector<double> v(fs.size());
        parallel_for(o.threads, fs.size(),
                     [&](size_t j) { v[j] = loss3(o, *fs[j].f, x, fs[j].m, fs[j].k); });
        if (strict) {
            double acc = 0.0;
            for (double t : v) acc += t;
            return acc;
        }
        DD acc;
        for (double t : v) acc.add(t);
        return acc.value();
    };
    auto f_and_grad = [&](double x, double& grad) {  // :228-240 with Loss5 :92-115
        const double h = 1e-6;                        // kNumericDiffStep, core_private.hpp:38
        std::vector<double> v(fs.size()), l(fs.size()), r(fs.size());
        parallel_for(o.threads, fs.size(), [&](size_t j) {
            const FrameState& s = fs[j];
            std::vector<double> P((size_t)s.f->n * 3);
            double g[3];
            problem_matrix(o, *s.f, x, P.data());
            v[j] = o.simplified ? loss_rows_P(P.data(), s.f->n, s.f->order.data(), s.k)
                   : strict     ? orc_strict::loss5_P(P.data(), s.f->n, s.m, s.k, g)
                                : loss5_P(P.data(), s.f->n, s.f->order.data(), s.m, s.k, g);
            l[j] = loss3(o, *s.f, x - h, s.m, s.k);
            r[j] = loss3(o, *s.f, x + h, s.m, s.k);
        });
        if (strict) {
            double av = 0.0, ag = 0.0;
            for (size_t j = 0; j < fs.size(); ++j) { av += v[j]; ag += (r[j] - l[j]) / 2 / h; }
            grad = ag;
            return av;
        }
        DD av, ag;
        for (size_t j = 0; j < fs.size(); ++j) {
            av.add(v[j]);
            ag.add((r[j] - l[j]) / 2 / h);  // :112
        }
        grad = ag.value();
        return av.value();
    };

    const double delay_b = 0.3;  // :260
    double delay_v = 0.0;        // :261 (zero-initialised)
    int converge_counter = 0;
    for (int it = 0; it < 400; ++it) {  // :309
        n_outer++;
        // do_opt_motion, :262-296
        std::vector<LbfgsStats> st(fs.size());
        if (!o.simplified) parallel_for(o.threads, fs.size(), [&](size_t j) {
            FrameState& s = fs[j];
            std::vector<double> P((size_t)s.f->n * 3);
            problem_matrix(o, *s.f, delay, P.data());
            const int n = s.f->n;
            const double k = s.k;
            if (strict)
                lbfgs3([&](const double* x, double* g) { return orc_strict::loss5_P(P.data(), n, x, k, g); },
                       s.m, &st[j], DotStrict());
            else
                lbfgs3([&](const double* x, double* g) { return loss5_P(P.data(), n, s.f->order.data(), x, k, g); }, s.m,
                       &st[j]);
        });
        for (auto& t : st) { n_lbfgs_eval += t.evals; n_lbfgs_iter += t.iters; }
        n_build += (long)fs.size();
        // do_opt_delay, :298-305, Backtrack::Step backtrack.cpp:3-13, hyper :226
        const double x0 = delay - delay_b * delay_v;
        double p;
        const double v = f_and_grad(x0, p);
        n_build += 3 * (long)fs.size();
        const double mm = p * p;
        double t = 1e-3;
        for (int i = 0; i < 10; ++i) {
            double v1 = sum_loss3(x0 - t * p);
            n_build += (long)fs.size();
            if (v - v1 >= t * 2e-4 * mm) break;
            t *= .1;
        }
        const double step = -t * p;
        delay_v = delay_b * delay_v + step;
        delay += delay_v;
        const double step_size = std::fabs(step);
        if (trace && trace->n < trace->cap) {
            trace->delays[trace->n] = delay;
            trace->steps[trace->n] = step_size;
            trace->n++;
        }
        if (step_size < 1e-4) converge_counter++; else converge_counter = 0;  // :316-320
        if (converge_counter > 5) break;                                       // :322
        if (std::fabs(delay - center) > radius) break;                         // :326
    }
    *out_cost = sum_loss3(delay);  // :333
    *out_delay = delay;
    if (counters) {
        counters[0] = n_outer; counters[1] = n_build; counters[2] = n_lbfgs_eval;
        counters[3] = n_lbfgs_iter; counters[4] = (long)fs.size();
    }
    return OK;
}

}  // namespace

// =============================================================================================
extern "C" {

void* orc_create() { return new Oracle(); }
void orc_destroy(void* h) { delete (Oracle*)h; }
const char* orc_last_error(void* h) { return ((Oracle*)h)->err.c_str(); }
void orc_set_threads(void* h, int t) { ((Oracle*)h)->threads = t < 1 ? 1 : t; }
void orc_set_strict(void* h, int strict, const int64_t* frame_order, int n) {
    Oracle& o = *(Oracle*)h;
    o.strict = strict != 0;
    o.frame_order.assign(frame_order, frame_order + (frame_order ? n : 0));
}
void orc_set_loss_mode(void* h, int simplified) { ((Oracle*)h)->simplified = simplified != 0; }
void orc_set_rng(void* h, uint64_t seed, uint64_t call_no) {
    ((Oracle*)h)->seed = seed;
    ((Oracle*)h)->call_no = call_no;
}
uint64_t orc_call_no(void* h) { return ((Oracle*)h)->call_no; }

// SetGyroQuaternions, fixed rate (core_private.cpp:135-140)
int orc_set_gyro_fixed(void* h, const double* quats, size_t count, double sample_rate,
                       double first_timestamp) {
    Oracle& o = *(Oracle*)h;
    if (count < 2) { o.err = "need at least 2 quaternions"; return E_INVALID; }
    o.sr = sample_rate;
    o.q0 = first_timestamp;
    o.resampled.assign(quats, quats + 4 * count);
    build_spline(o, quats, (long)count);
    return OK;
}

// SetGyroQuaternions, variable rate (core_private.cpp:142-190)
int orc_set_gyro_var(void* h, const int64_t* ts, const double* quats, size_t count) {
    Oracle& o = *(Oracle*)h;
    if (count < 2) { o.err = "need at least 2 quaternions"; return E_INVALID; }
    const uint64_t k_uhz_in_hz = 1000000ULL, k_us_in_sec = 1000000ULL;
    uint64_t span = (uint64_t)(ts[count - 1] - ts[0]);
    if (span == 0) { o.err = "set-gyro-quaternions: zero time span"; return E_INVALID; }
    uint64_t actual_sr_uhz = k_uhz_in_hz * k_us_in_sec * (uint64_t)count / span;  // :146-147
    int sr_hz = int(std::round((double)actual_sr_uhz / 50. / (double)k_uhz_in_hz) * 50);  // :148-149
    if (sr_hz <= 0) { o.err = "set-gyro-quaternions: sample rate rounds to zero"; return E_INVALID; }
    std::vector<uint64_t> nts;
    const uint64_t last = (uint64_t)ts[count - 1];
    // :152-155 — first index by unsigned integer division (the ceil() is a no-op)
    int sample = (int)std::ceil((double)((uint64_t)(ts[0] * (int64_t)sr_hz) / k_us_in_sec));
    for (; k_us_in_sec * (uint64_t)sample / (uint64_t)sr_hz < last; sample += 1)
        nts.push_back(k_us_in_sec * (uint64_t)sample / (uint64_t)sr_hz);
    for (size_t i = 1; i < count; ++i) {  // :157-164
        if (ts[i - 1] > ts[i]) {
            o.err = "set-gyro-quaternions:  timestamps out of order at pos " + std::to_string(i) +
                    " (" + std::to_string(ts[i - 1]) + " > " + std::to_string(ts[i]) + ")";
            return E_ORDER;
        }
    }
    if (nts.size() < 2) { o.err = "set-gyro-quaternions: fewer than 2 resampled samples"; return E_INVALID; }
    std::vector<double> nq(4 * nts.size());
    for (size_t i = 0; i < nts.size(); ++i) {  // :166-182
        uint64_t t = nts[i];
        size_t idx = std::lower_bound(ts, ts + count, t,
                                      [](int64_t a, uint64_t b) { return (uint64_t)a < b; }) - ts;
        if (idx > 0) {
            double u = 1. * (double)(t - (uint64_t)ts[idx - 1]) / (double)(ts[idx] - ts[idx - 1]);
            slerp(quats + 4 * (idx - 1), quats + 4 * idx, u, &nq[4 * i], !o.strict);
        } else {
            for (int c = 0; c < 4; ++c) nq[4 * i + c] = quats[4 * idx + c];
        }
        if (!all_finite(&nq[4 * i], 4)) {
            o.err = "set-gyro-quaternions: non-finite sample after interpolation";
            return E_NONFINITE;
        }
    }
    o.sr = 1. * sr_hz;                               // :183
    o.q0 = 1. * (double)nts[0] / (double)k_us_in_sec;  // :184
    o.resampled = nq;
    build_spline(o, nq.data(), (long)nts.size());
    return OK;
}

// SetTrackResult (core_private.cpp:192-203); copies the caller's buffers.
int orc_set_track(void* h, int64_t frame, const double* ts_a, const double* ts_b,
                  const double* rays_a, const double* rays_b, size_t count) {
    Oracle& o = *(Oracle*)h;
    const char* names[4] = {"rays_a", "rays_b", "ts_a", "ts_b"};
    const double* ptr[4] = {rays_a, rays_b, ts_a, ts_b};
    const size_t len[4] = {3 * count, 3 * count, count, count};
    for (int i = 0; i < 4; ++i)
        if (!all_finite(ptr[i], len[i])) {
            o.err = std::string("set-track-result: non-finite numbers in ") + names[i];
            return E_NONFINITE;
        }
    Frame& f = o.frames[frame];
    f.n = (int)count;
    f.ts_a.assign(ts_a, ts_a + count);
    f.ts_b.assign(ts_b, ts_b + count);
    f.ra.assign(rays_a, rays_a + 3 * count);
    f.rb.assign(rays_b, rays_b + 3 * count);
    f.order.resize(count);
    for (size_t i = 0; i < count; ++i) f.order[i] = (int)i;
    std::sort(f.order.begin(), f.order.end(), [&](int a, int b) {
        return f.ts_a[a] < f.ts_a[b] || (f.ts_a[a] == f.ts_a[b] && a < b);
    });
    return OK;
}

// generic grid (extension used by the sharded path and the tests)
int orc_presync_grid(void* h, int64_t fb, int64_t fe, const double* delays, int n, uint64_t stream,
                     uint64_t call_no, uint64_t idx_base, double* costs, double* frame_costs,
                     int* flags) {
    return presync_grid(*(Oracle*)h, fb, fe, delays, n, stream, call_no, idx_base, costs,
                        frame_costs, flags);
}

// delay grid of pre_sync's loop (core_private.cpp:69-70), fp accumulation included
int orc_presync_delays(double initial, double step, double radius, double* out, int cap) {
    int n = 0;
    for (double d = initial - radius; d < initial + radius; d += step) {
        if (out && n < cap) out[n] = d;
        n++;
        if (n > (1 << 28)) break;
    }
    return n;
}

// PreSync (core_private.cpp:205-209 -> pre_sync :61-90).  Returns {cost, delay} of the
// lexicographically smallest (cost, delay) pair (:89).
int orc_presync(void* h, double initial, int64_t fb, int64_t fe, double step, double radius,
                double* out_cost, double* out_delay) {
    Oracle& o = *(Oracle*)h;
    int n = orc_presync_delays(initial, step, radius, nullptr, 0);
    std::vector<double> delays(n), costs(n);
    orc_presync_delays(initial, step, radius, delays.data(), n);
    uint64_t call = o.call_no++;
    int flags = 0;
    int rc = presync_grid(o, fb, fe, delays.data(), n, kStreamPreSync, call, 0, costs.data(),
                          nullptr, &flags);
    if (rc) return rc;
    if (flags) {  // :76-83
        o.err = (flags & 1) ? "pre-sync: non-finite numbers in P"
              : (flags & 2) ? "pre-sync: non-finite numbers in M"
              : (flags & 4) ? "pre-sync: non-finite r" : "pre-sync: non-finite rho";
        return E_NONFINITE;
    }
    if (n == 0) { o.err = "pre-sync: empty delay grid"; return E_INVALID; }
    int best = 0;
    for (int i = 1; i < n; ++i)
        if (costs[i] < costs[best] || (costs[i] == costs[best] && delays[i] < delays[best])) best = i;
    *out_cost = costs[best];
    *out_delay = delays[best];
    return OK;
}

// DebugPreSync (core_private.cpp:336-361): linspace grid, no panics
int orc_debug_presync(void* h, double initial, int64_t fb, int64_t fe, double radius,
                      double* delays, double* costs, int point_count) {
    Oracle& o = *(Oracle*)h;
    for (int i = 0; i < point_count; ++i)
        delays[i] = initial - radius + 2 * radius * i / (point_count - 1);  // :345
    uint64_t call = o.call_no++;
    return presync_grid(o, fb, fe, delays, point_count, kStreamDebugPreSync, call, 0, costs, nullptr,
                        nullptr);
}

// Sync (core_private.cpp:211-334)
int orc_sync(void* h, double initial, int64_t fb, int64_t fe, double center, double radius,
             double* out_cost, double* out_delay) {
    Oracle& o = *(Oracle*)h;
    uint64_t call = o.call_no++;
    return sync_impl(o, initial, fb, fe, center, radius, call, out_cost, out_delay, nullptr, nullptr);
}
int orc_sync_traced(void* h, double initial, int64_t fb, int64_t fe, double center, double radius,
                    double* out_cost, double* out_delay, double* tr_delays, double* tr_steps,
                    int cap, int* n_trace, long* counters) {
    Oracle& o = *(Oracle*)h;
    uint64_t call = o.call_no++;
    SyncTrace tr{tr_delays, tr_steps, cap, 0};
    int rc = sync_impl(o, initial, fb, fe, center, radius, call, out_cost, out_delay, &tr, counters);
    if (n_trace) *n_trace = tr.n;
    return rc;
}

// ---- stage probes (used by the stage-level parity tests) -------------------------------------
long orc_gyro_count(void* h) { return ((Oracle*)h)->nq; }
double orc_gyro_rate(void* h) { return ((Oracle*)h)->sr; }
double orc_gyro_start(void* h) { return ((Oracle*)h)->q0; }
void orc_get_spline(void* h, double* rec) {
    Oracle& o = *(Oracle*)h;
    std::copy(o.rec.begin(), o.rec.end(), rec);
}
void orc_get_resampled(void* h, double* q) {
    Oracle& o = *(Oracle*)h;
    std::copy(o.resampled.begin(), o.resampled.end(), q);
}
void orc_spline_eval(void* h, const double* x, int n, double* out) {
    Oracle& o = *(Oracle*)h;
    for (int i = 0; i < n; ++i) spline_eval4(o.rec.data(), o.nq, x[i], out + 4 * i);
}
int orc_problem_matrix(void* h, int64_t frame, double delay, double* P) {
    Oracle& o = *(Oracle*)h;
    auto it = o.frames.find(frame);
    if (it == o.frames.end()) { o.err = "no such frame"; return E_INVALID; }
    problem_matrix(o, it->second, delay, P);
    return OK;
}
// RANSAC on frame's P(delay) with an explicit RNG key tuple
int orc_guess_motion(void* h, int64_t frame, double delay, int iters, uint64_t stream,
                     uint64_t call_no, uint64_t offset_idx, double* m, double* k) {
    Oracle& o = *(Oracle*)h;
    auto it = o.frames.find(frame);
    if (it == o.frames.end()) { o.err = "no such frame"; return E_INVALID; }
    const Frame& f = it->second;
    std::vector<double> P((size_t)f.n * 3), nP, r2;
    problem_matrix(o, f, delay, P.data());
    guess_motion(P.data(), f.n, iters, rng_task_key(o.seed, stream, call_no, offset_idx, frame), m,
                 nP, r2, o.strict);
    if (k) *k = o.strict ? clamp_k(1 / orc_strict::norm_PM(P.data(), f.n, m) * 1e2)
                         : clamp_k(1.0 / norm_PM(P.data(), f.n, f.order.data(), m) * 1e2);
    return OK;
}
// guess_motion's spec-mode loop with every hypothesis kept: v_out[3 t..3 t + 2] the hypothesis of
// iteration t, q_out[t] its exact quartile r2[n/4], *best the index of the first strict minimum (the
// one guess_motion returns).  Lets the tests check what a frame built to tie actually ties.
int orc_estimator_trace(void* h, int64_t frame, double delay, int iters, uint64_t stream,
                        uint64_t call_no, uint64_t offset_idx, double* v_out, double* q_out, int* best) {
    Oracle& o = *(Oracle*)h;
    auto it = o.frames.find(frame);
    if (it == o.frames.end()) { o.err = "no such frame"; return E_INVALID; }
    const Frame& f = it->second;
    const int n = f.n;
    std::vector<double> P((size_t)n * 3), nP((size_t)n * 3), r2(n);
    problem_matrix(o, f, delay, P.data());
    const uint64_t key = rng_task_key(o.seed, stream, call_no, offset_idx, frame);
    for (int i = 0; i < n; ++i) safe_normalize3(&P[3 * i], &nP[3 * i]);
    double least = std::numeric_limits<double>::infinity();
    *best = 0;
    for (int t = 0; t < iters; ++t) {
        uint32_t a = rng_index(key, t, 0, n);
        uint32_t b, k = 1;
        do { b = rng_index(key, t, k++, n); } while (b == a);
        const double* pa = &P[3 * a];
        const double* pb = &P[3 * b];
        double c[3] = {hyp_cross_term(pa[1], pb[2], pa[2] * pb[1]), hyp_cross_term(pa[2], pb[0], pa[0] * pb[2]),
                       hyp_cross_term(pa[0], pb[1], pa[1] * pb[0])};
        double* v = v_out + 3 * t;
        safe_normalize3(c, v);
        for (int i = 0; i < n; ++i) {
            double r = dot3(&nP[3 * i], v);
            r2[i] = r * r;
        }
        std::nth_element(r2.begin(), r2.begin() + n / 4, r2.end());
        q_out[t] = r2[n / 4];
        if (q_out[t] < least) { least = q_out[t]; *best = t; }
    }
    return OK;
}
int orc_loss3(void* h, int64_t frame, double delay, const double* m, double k, double* out) {
    Oracle& o = *(Oracle*)h;
    auto it = o.frames.find(frame);
    if (it == o.frames.end()) return E_INVALID;
    *out = loss3(o, it->second, delay, m, k);
    return OK;
}
int orc_loss5(void* h, int64_t frame, double delay, const double* m, double k, double* out,
              double* grad) {
    Oracle& o = *(Oracle*)h;
    auto it = o.frames.find(frame);
    if (it == o.frames.end()) return E_INVALID;
    std::vector<double> P((size_t)it->second.n * 3);
    problem_matrix(o, it->second, delay, P.data());
    *out = o.strict ? orc_strict::loss5_P(P.data(), it->second.n, m, k, grad)
                    : loss5_P(P.data(), it->second.n, it->second.order.data(), m, k, grad);
    return OK;
}
int orc_lbfgs(void* h, int64_t frame, double delay, double* m, double k, double* fout, int* iters,
              int* evals) {
    Oracle& o = *(Oracle*)h;
    auto it = o.frames.find(frame);
    if (it == o.frames.end()) return E_INVALID;
    const Frame& f = it->second;
    std::vector<double> P((size_t)f.n * 3);
    problem_matrix(o, f, delay, P.data());
    LbfgsStats st;
    double v = lbfgs3([&](const double* x, double* g) { return loss5_P(P.data(), f.n, f.order.data(), x, k, g); }, m, &st);
    if (fout) *fout = v;
    if (iters) *iters = st.iters;
    if (evals) *evals = st.evals;
    return OK;
}
// optdata_fill_gyro, core_testcode.cpp:37-53 (the caller-side gyro integration), with the
// gyro_orientation axis mapping of the product documented in include/rssync_b200.h
int orc_integrate_gyro(const double* ts, const double* gyro, size_t count, const char* orient, double* out) {
    int src[3] = {0, 1, 2};
    double sgn[3] = {1, 1, 1};
    if (orient) {
        if (std::string(orient).size() != 3) return 1;
        for (int i = 0; i < 3; ++i) {
            const char c = orient[i];
            const std::string axes = "xyzXYZ";
            const size_t at = axes.find(c);
            if (at == std::string::npos) return 1;
            src[i] = (int)(at % 3);
            sgn[i] = at < 3 ? -1.0 : 1.0;
        }
    }
    // The contract's order of operations (shared with the engine, host and device): the recurrence
    // q_i = normalise(d_i (x) q_{i-1}) runs inside blocks of 512 samples, each from the identity; the
    // blocks' last values are chained into per-block prefixes; every sample is then its block-local
    // value times its block's prefix, normalised.  (The reference's caller runs one sequential
    // recurrence, core_testcode.cpp:41-46; the two differ by rounding only.)
    const size_t B = 512;
    auto increment = [&](size_t i, double d[4]) {  // quat_from_aa(w_i dt_i), quat.cpp:5-17; d_0 = identity
        if (i == 0) { d[0] = 1.; d[1] = d[2] = d[3] = 0.; return; }
        const double dt = ts[i] - ts[i - 1];                            // :44
        double aa[3];
        for (int c = 0; c < 3; ++c) aa[c] = sgn[c] * gyro[3 * i + src[c]] * dt;
        const double theta_squared = (aa[0] * aa[0] + aa[1] * aa[1]) + aa[2] * aa[2];  // quat.cpp:6
        if (theta_squared > 0.) {                                        // quat.cpp:8-12
            const double theta = std::sqrt(theta_squared);
            const double half_theta = theta * 0.5;
            const double k = orc::spec_sin(half_theta) / theta;
            d[0] = orc::spec_cos(half_theta); d[1] = aa[0] * k; d[2] = aa[1] * k; d[3] = aa[2] * k;
        } else {                                                         // quat.cpp:13-16
            d[0] = 1.; d[1] = aa[0] * 0.5; d[2] = aa[1] * 0.5; d[3] = aa[2] * 0.5;
        }
    };
    auto mul_norm = [](const double* p, const double* q, double* out) {  // normalise(p (x) q), quat.cpp:34-37
        const double r0 = ((p[0] * q[0] - p[1] * q[1]) - p[2] * q[2]) - p[3] * q[3];
        const double r1 = ((p[0] * q[1] + p[1] * q[0]) + p[2] * q[3]) - p[3] * q[2];
        const double r2 = ((p[0] * q[2] - p[1] * q[3]) + p[2] * q[0]) + p[3] * q[1];
        const double r3 = ((p[0] * q[3] + p[1] * q[2]) - p[2] * q[1]) + p[3] * q[0];
        const double nrm = std::sqrt(((r0 * r0 + r1 * r1) + r2 * r2) + r3 * r3);
        out[0] = r0 / nrm; out[1] = r1 / nrm; out[2] = r2 / nrm; out[3] = r3 / nrm;  // :45
    };
    const double ident[4] = {1., 0., 0., 0.};
    const size_t nb = (count + B - 1) / B;
    std::vector<double> local(4 * count), prefix(4 * (nb + 1));
    for (size_t b = 0; b < nb; ++b) {
        const double* prev = ident;
        for (size_t i = b * B; i < std::min(count, (b + 1) * B); ++i) {
            double d[4];
            increment(i, d);
            mul_norm(d, prev, &local[4 * i]);
            prev = &local[4 * i];
        }
    }
    for (int c = 0; c < 4; ++c) prefix[c] = ident[c];
    for (size_t b = 0; b < nb; ++b) mul_norm(&local[4 * (std::min(count, (b + 1) * B) - 1)], &prefix[4 * b], &prefix[4 * (b + 1)]);
    for (size_t i = 0; i < count; ++i) mul_norm(&local[4 * i], &prefix[4 * (i / B)], out + 4 * i);
    return 0;
}

void orc_log1p(const double* x, int n, double* out) {
    for (int i = 0; i < n; ++i) out[i] = log1p_nonneg(x[i]);
}
void orc_slerp(const double* p, const double* q, double t, double* out) { slerp(p, q, t, out); }
void orc_slerp_spec(const double* p, const double* q, double t, double* out) { slerp(p, q, t, out, true); }
// which: 0 sin, 1 cos, 2 acos of the contract
void orc_spec_trig(const double* x, int n, int which, double* out) {
    for (int i = 0; i < n; ++i) out[i] = which == 0 ? orc::spec_sin(x[i]) : which == 1 ? orc::spec_cos(x[i]) : orc::spec_acos(x[i]);
}
uint32_t orc_rng_index(uint64_t seed, uint64_t stream, uint64_t call_no, uint64_t offset_idx,
                       int64_t frame, uint32_t iter, uint32_t k, uint32_t n) {
    return rng_index(rng_task_key(seed, stream, call_no, offset_idx, frame), iter, k, n);
}
double orc_ddsum(const double* x, int n) {
    DD a;
    for (int i = 0; i < n; ++i) a.add(x[i]);
    return a.value();
}
int orc_has_hw_fma() {
#ifdef __FMA__
    return 1;
#else
    return 0;
#endif
}

}  // extern "C"
