// The two per-sample operations of the gyro integration (optdata_fill_gyro, core_testcode.cpp:37-53),
// written once for the host (host_ingest.cpp) and the device (engine.cu) so that both produce the
// same bits: the increment d_i = quat_from_aa(w_i (t_i - t_{i-1})) (quat.cpp:5-17, with the
// contract's sin / cos) and q = normalise(p (x) q) (quat.cpp:33-38 + arma::normalise).
#pragma once
#include <cstddef>

#include "spec_trig.h"

namespace rs {

constexpr size_t kGyroScanBlock = 512;  // samples per block of the blocked recurrence

// The gyro axis mapping is a 3x3 row-major matrix m: the angular velocity in the integration's frame
// is w = m g.  Its arithmetic (part of the contract, DESIGN.md section 3.8): w_c sums m[3c+j] g_j over
// the j with m[3c+j] != 0 only; the first kept term is the product, the others are added to it left to
// right, without contraction; a row without a non-zero coefficient gives w_c = +0.0.  A signed
// permutation matrix therefore gives w_c = (+-1 g_src) bit for bit, the sign of a zero and a NaN or inf
// on an axis it does not read included.
RS_TRIG_HD double gyro_map_row(const double* row, const double* g) {
    double w = 0.0;
    bool kept = false;
    for (int j = 0; j < 3; ++j)
        if (row[j] != 0.0) {
            const double t = row[j] * g[j];
            w = kept ? w + t : t;
            kept = true;
        }
    return w;
}

// d_0 = identity; d_i = quat_from_aa((m g_i) (t_i - t_{i-1}))
RS_TRIG_HD void gyro_increment(const double* ts, const double* gyro, size_t i, const double m[9], double d[4]) {
    if (i == 0) { d[0] = 1.0; d[1] = 0.0; d[2] = 0.0; d[3] = 0.0; return; }
    const double dt = ts[i] - ts[i - 1];
    const double* g = gyro + 3 * i;
    const double a0 = gyro_map_row(m, g) * dt, a1 = gyro_map_row(m + 3, g) * dt, a2 = gyro_map_row(m + 6, g) * dt;
    const double th2 = (a0 * a0 + a1 * a1) + a2 * a2;
    if (th2 > 0.) {
        const double th = trig_detail::sqrt_(th2), half = th * 0.5, k = spec_sin(half) / th;
        d[0] = spec_cos(half); d[1] = a0 * k; d[2] = a1 * k; d[3] = a2 * k;
    } else {
        d[0] = 1.; d[1] = a0 * 0.5; d[2] = a1 * 0.5; d[3] = a2 * 0.5;
    }
}

RS_TRIG_HD void quat_mul_normalise(const double* p, const double* q, double* out) {
    const double r0 = ((p[0] * q[0] - p[1] * q[1]) - p[2] * q[2]) - p[3] * q[3];
    const double r1 = ((p[0] * q[1] + p[1] * q[0]) + p[2] * q[3]) - p[3] * q[2];
    const double r2 = ((p[0] * q[2] - p[1] * q[3]) + p[2] * q[0]) + p[3] * q[1];
    const double r3 = ((p[0] * q[3] + p[1] * q[2]) - p[2] * q[1]) + p[3] * q[0];
    const double nrm = trig_detail::sqrt_(((r0 * r0 + r1 * r1) + r2 * r2) + r3 * r3);
    out[0] = r0 / nrm; out[1] = r1 / nrm; out[2] = r2 / nrm; out[3] = r3 / nrm;
}

// quat_slerp, quat.cpp:55-74, with the contract's acos / sin
RS_TRIG_HD void quat_slerp_spec(const double* p, const double* q_in, double t, double* out) {
    double q[4] = {q_in[0], q_in[1], q_in[2], q_in[3]};
    double cosang = ((p[0] * q[0] + p[1] * q[1]) + p[2] * q[2]) + p[3] * q[3];
    if (cosang < 0) {
        q[0] = -q[0]; q[1] = -q[1]; q[2] = -q[2]; q[3] = -q[3];
        cosang = ((p[0] * q[0] + p[1] * q[1]) + p[2] * q[2]) + p[3] * q[3];
    }
    const double ang = spec_acos(cosang);
    double wp, wq;
    if (ang > 1e-9) {
        const double s = spec_sin(ang);
        wp = spec_sin((1 - t) * ang) / s;
        wq = spec_sin(t * ang) / s;
    } else {
        wp = 1 - t;
        wq = t;
    }
    for (int c = 0; c < 4; ++c) out[c] = wp * p[c] + wq * q[c];
}

}  // namespace rs
