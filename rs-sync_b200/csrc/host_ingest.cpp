// Host-side gyro ingest of the engine: variable-rate resampling and the natural-cubic-spline
// coefficient build.  Both are short sequential recurrences over the gyro track (O(n), run once
// per SetGyroQuaternions call, ~1 ms for a minute of 1 kHz data), and their results feed the
// finite-difference delay gradient of Sync, which amplifies 1-ulp differences by 1/(2h) = 5e5 —
// so they are evaluated in one fixed order on the host and only the finished 128-byte spline
// records travel to the GPU (DESIGN.md §4).  Compile with -ffp-contract=off.
#include "host_ingest.h"

#include "spec_trig.h"

#include <algorithm>
#include <cmath>
#include <memory>
#include <mutex>
#include <thread>

namespace rs {

namespace {

// ndspline::make (ndspline.cpp:13-19) = spline::set_points (minispline.cpp:3-46) per component:
// unit-spaced knots; interior rows [1/3, 4/3, 1/3] with rhs y[i+1] - 2 y[i] + y[i-1], natural
// boundary rows [., 2, 0] / [0, 2, .] with rhs 0; eliminate downwards (:22-26), then upwards
// (:28-32), divide (:34), then d and b per interval (:38-44).
//
// The matrix entries and both elimination factors do not depend on the data, only on n, so they are
// computed once for the four components -- by the same operations on the same values as the
// reference's per-component loop, hence the same bits.  The interior rows start out identical, so
// the elimination state reaches a floating-point fixed point after a few dozen rows; from there on
// every row repeats it exactly and the (division-bound) recurrence is not re-evaluated.  What
// remains sequential per component is rhs[i+1] -= rhs[i] * f[i] and its mirror image, which run
// for the four components side by side.
struct Elimination {
    std::vector<double> f_down;  // f_down[i]: factor with which row i is subtracted from row i + 1
    std::vector<double> f_up;    // f_up[i]:   factor with which row i is subtracted from row i - 1
    std::vector<double> diag;    // diagonal after both sweeps
};

Elimination eliminate(size_t n) {
    Elimination e;
    e.f_down.assign(n, 0.0);
    e.f_up.assign(n, 0.0);
    e.diag.assign(n, 2.0 / 3.0 * 2.0);
    std::vector<double> sub(n, 1.0 / 3.0), sup(n, 1.0 / 3.0);
    std::vector<double>& diag = e.diag;
    sub[0] = 0.0; diag[0] = 2.0; sup[0] = 0.0;
    sub[n - 1] = 0.0; diag[n - 1] = 2.0; sup[n - 1] = 0.0;
    // downwards, minispline.cpp:22-26: row i clears the sub-diagonal of row i + 1, for i + 2 < n
    size_t steady = n;  // rows steady .. n-2 leave this sweep in the same state
    for (size_t i = 0; i + 2 < n; ++i) {
        const double f = 1. / diag[i] * sub[i + 1];
        sub[i + 1] -= diag[i] * f;
        diag[i + 1] -= sup[i] * f;
        e.f_down[i] = f;
        // row i + 1 came out exactly like row i (both interior): the rows below start out like
        // row i + 1 did, so each repeats this step with the same operands
        if (i >= 1 && sub[i + 1] == sub[i] && diag[i + 1] == diag[i] && f == e.f_down[i - 1]) {
            for (size_t j = i + 1; j + 2 < n; ++j) {
                sub[j + 1] = sub[i];
                diag[j + 1] = diag[i];
                e.f_down[j] = f;
            }
            steady = i;
            break;
        }
    }
    // upwards, :28-32: row i clears the super-diagonal of row i - 1, for i > 1
    for (size_t i = n - 1; i > 1; --i) {
        const double f = 1. / diag[i] * sup[i - 1];
        diag[i - 1] -= sub[i] * f;
        sup[i - 1] -= diag[i] * f;
        e.f_up[i] = f;
        // rows i - 1 and i entered this sweep in the same state (both in the steady range, as is
        // row i + 1, whose sub-diagonal entered step i + 1) and row i - 1 left it with row i's
        // diagonal: step i - 1 therefore sees the operands of step i, and so on up to `steady`
        if (i + 1 <= n - 2 && i - 1 > steady && diag[i - 1] == diag[i]) {
            for (size_t j = i - 1; j > steady; --j) {  // step j writes row j - 1 >= steady
                diag[j - 1] = diag[i - 1];
                sup[j - 1] = sup[i - 1];
                e.f_up[j] = f;
            }
            i = steady + 1;  // the loop continues with step `steady`
        }
    }
    return e;
}

}  // namespace

void build_spline_system(const double* quats, size_t n, double* rhs, double* diag) {
    // the elimination only depends on n: the orientation search builds 48 splines of one length
    static std::mutex mu;
    static std::shared_ptr<const Elimination> cached;
    static size_t cached_n = 0;
    std::shared_ptr<const Elimination> ep;
    {
        std::lock_guard<std::mutex> lk(mu);
        if (cached && cached_n == n) ep = cached;
    }
    if (!ep) {
        ep = std::make_shared<const Elimination>(eliminate(n));
        std::lock_guard<std::mutex> lk(mu);
        cached = ep;
        cached_n = n;
    }
    const Elimination& e = *ep;
    std::copy(e.diag.begin(), e.diag.end(), diag);
    // right-hand sides of the four components, interleaved like the input; the downward sweep (:25)
    // consumes each row right after it is formed
    for (int c = 0; c < 4; ++c) rhs[c] = rhs[4 * (n - 1) + c] = 0.0;
    for (size_t i = 1; i + 1 < n; ++i) {
        const double f = e.f_down[i - 1];
        for (int c = 0; c < 4; ++c) {
            const double r = (quats[4 * (i + 1) + c] - 2 * quats[4 * i + c]) + quats[4 * (i - 1) + c];
            rhs[4 * i + c] = r - rhs[4 * (i - 1) + c] * f;
        }
    }
    for (size_t i = n - 1; i > 1; --i) {  // :31
        const double f = e.f_up[i];
        for (int c = 0; c < 4; ++c) rhs[4 * (i - 1) + c] -= rhs[4 * i + c] * f;
    }
}

bool parse_orientation(const char* orient, double m[9]) {
    for (int k = 0; k < 9; ++k) m[k] = (k % 4 == 0) ? 1.0 : 0.0;
    if (!orient) return true;
    for (int i = 0; i < 3; ++i) {
        const char ch = orient[i];
        const char lo = (char)(ch | 0x20);
        if (lo < 'x' || lo > 'z') return false;
        m[3 * i + 0] = m[3 * i + 1] = m[3 * i + 2] = 0.0;
        m[3 * i + (lo - 'x')] = (ch == lo) ? -1.0 : 1.0;
    }
    return orient[3] == 0;
}

void integrate_gyro(const double* ts, const double* gyro, size_t count, const double m[9], double* out) {
    if (count == 0) return;
    // The contract's order of operations (the device kernels of engine.cu follow the same one, see
    // gyro_local_kernel): the recurrence runs inside blocks of kGyroScanBlock samples, each from the
    // identity; the blocks' last values are chained into per-block prefixes; every sample is its
    // block-local value times its block's prefix, normalised.
    const size_t B = kGyroScanBlock;
    const size_t nb = (count + B - 1) / B;
    std::vector<double> local(4 * count), prefix(4 * (nb + 1));
    const double ident[4] = {1.0, 0.0, 0.0, 0.0};
    for (size_t b = 0; b < nb; ++b) {
        const double* prev = ident;
        for (size_t i = b * B; i < std::min(count, (b + 1) * B); ++i) {
            double d[4];
            gyro_increment(ts, gyro, i, m, d);
            quat_mul_normalise(d, prev, &local[4 * i]);
            prev = &local[4 * i];
        }
    }
    for (int c = 0; c < 4; ++c) prefix[c] = ident[c];
    for (size_t b = 0; b < nb; ++b)
        quat_mul_normalise(&local[4 * (std::min(count, (b + 1) * B) - 1)], &prefix[4 * b], &prefix[4 * (b + 1)]);
    for (size_t i = 0; i < count; ++i) quat_mul_normalise(&local[4 * i], &prefix[4 * (i / B)], out + 4 * i);
}

// SyncProblemPrivate::SetGyroQuaternions(const int64_t*, const double*, size_t),
// core_private.cpp:142-190, integer quirks included (see SURVEY.md section 8 a3): everything of it that
// does not touch the samples -- the rate, the uniform integer-microsecond grid, the order check.  The
// per-sample half (lower_bound + slerp, :166-182) runs on the device (resample_kernel, engine.cu).
IngestStatus plan_variable_rate(const int64_t* ts_us, size_t count, ResamplePlan& plan, std::string& err) {
    constexpr uint64_t kMicro = 1000000ULL;
    if (count < 2) { err = "set-gyro-quaternions: need at least 2 samples"; return IngestStatus::Invalid; }
    const uint64_t span = (uint64_t)(ts_us[count - 1] - ts_us[0]);
    if (span == 0) { err = "set-gyro-quaternions: zero time span"; return IngestStatus::Invalid; }
    const uint64_t rate_uhz = kMicro * kMicro * (uint64_t)count / span;                   // :146-147
    const int rate_hz = int(std::round((double)rate_uhz / 50. / (double)kMicro) * 50);   // :148-149
    if (rate_hz <= 0) { err = "set-gyro-quaternions: sample rate rounds to zero"; return IngestStatus::Invalid; }
    const uint64_t t_last = (uint64_t)ts_us[count - 1];
    const int tick0 = (int)std::ceil((double)((uint64_t)(ts_us[0] * (int64_t)rate_hz) / kMicro));  // :152
    // grid point j is kMicro (tick0 + j) / rate_hz (integer division), for as long as it is < t_last (:153):
    // the count follows from the monotonicity of the quotient
    uint64_t n_out = 0;
    if (kMicro * (uint64_t)tick0 / (uint64_t)rate_hz < t_last) {
        // largest tick with kMicro tick / rate < t_last  <=>  kMicro tick < t_last rate  <=>  tick <= (t_last rate - 1) / kMicro
        const uint64_t last_tick = (t_last * (uint64_t)rate_hz - 1) / kMicro;
        n_out = last_tick - (uint64_t)tick0 + 1;
    }
    for (size_t i = 1; i < count; ++i) {  // :157-164
        if (ts_us[i - 1] > ts_us[i]) {
            err = "set-gyro-quaternions:  timestamps out of order at pos " + std::to_string(i) + " (" +
                  std::to_string(ts_us[i - 1]) + " > " + std::to_string(ts_us[i]) + ")";
            return IngestStatus::OutOfOrder;
        }
    }
    if (n_out < 2) { err = "set-gyro-quaternions: fewer than 2 resampled samples"; return IngestStatus::Invalid; }
    if (n_out > (uint64_t)INT32_MAX) { err = "set-gyro-quaternions: too many samples"; return IngestStatus::Invalid; }
    plan.rate_hz = (unsigned)rate_hz;
    plan.tick0 = (uint64_t)tick0;
    plan.n_out = (size_t)n_out;
    plan.sample_rate = 1. * rate_hz;                                                              // :183
    plan.first_timestamp = 1. * (double)(kMicro * (uint64_t)tick0 / (uint64_t)rate_hz) / (double)kMicro;  // :184
    if (!std::isfinite(plan.sample_rate)) { err = "set-gyro-quaternions: non-finite sample rate. wtf?"; return IngestStatus::NonFinite; }
    if (!std::isfinite(plan.first_timestamp)) { err = "set-gyro-quaternions: non-finite first timestamp. wtf?"; return IngestStatus::NonFinite; }
    return IngestStatus::Ok;
}

std::shared_ptr<const SplineElimination> spline_elimination(size_t n) {
    static std::mutex mu;
    static std::shared_ptr<const SplineElimination> cached;
    std::lock_guard<std::mutex> lk(mu);
    if (!cached || cached->f_down.size() != n) {
        Elimination e = eliminate(n);
        auto se = std::make_shared<SplineElimination>();
        se->f_down = std::move(e.f_down);
        se->f_up = std::move(e.f_up);
        se->diag = std::move(e.diag);
        cached = se;
    }
    return cached;
}

}  // namespace rs
