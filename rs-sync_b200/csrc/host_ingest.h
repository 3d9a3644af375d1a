// Host-side gyro ingest (see host_ingest.cpp).
#pragma once
#include <cstddef>
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

#include "gyro_scan.h"

namespace rs {

enum class IngestStatus { Ok = 0, Invalid = 1, NonFinite = 2, OutOfOrder = 3 };

// ndspline::make (ndspline.cpp:13-19), the sequential half: the tridiagonal system of the natural
// cubic spline on unit knots (minispline.cpp:3-32) for the four quaternion components, eliminated
// downwards and upwards.  rhs (4 n doubles, interleaved like the input) and diag (n doubles) are what
// is left of it: the second-derivative coefficient of sample i, component c is rhs[4 i + c] / diag[i]
// (:34).  The divisions and the b / d coefficients (:38-44) are independent per sample and are
// finished on the device (launch_spline_finish, engine.h).
void build_spline_system(const double* quats, size_t n, double* rhs /* 4 n */, double* diag /* n */);

// variable-rate SetGyroQuaternions (core_private.cpp:142-190), the part that does not touch the
// samples: output rate, the uniform integer-microsecond grid (point j = 1e6 (tick0 + j) / rate_hz in
// integer division, n_out points), quats_start, the order check.  The samples are interpolated on
// the device (launch_gyro_resample).
struct ResamplePlan {
    unsigned rate_hz = 0;
    uint64_t tick0 = 0;
    size_t n_out = 0;
    double sample_rate = 0.0, first_timestamp = 0.0;
};
IngestStatus plan_variable_rate(const int64_t* ts_us, size_t count, ResamplePlan& plan, std::string& err);

// the data-independent part of the spline system of n knots (elimination factors of both sweeps and
// the diagonal they leave), cached for the most recent n
struct SplineElimination {
    std::vector<double> f_down, f_up, diag;
};
std::shared_ptr<const SplineElimination> spline_elimination(size_t n);

// gyro_orientation string (null: "XYZ") -> its signed permutation matrix m (3x3 row-major, w = m g):
// character i names the input axis routed to output axis i, lower case flips its sign.  False if
// malformed.
bool parse_orientation(const char* orient, double m[9]);

// optdata_fill_gyro (core_testcode.cpp:37-53), the step before SetGyroQuaternions: q_0 = identity,
// q_i = normalise(quat_from_aa(w_i (t_i - t_{i-1})) (x) q_{i-1}) (quat.cpp:5-17, 33-38), with
// w_i = m g_i under the mapping arithmetic of gyro_scan.h (gyro_map_row).
// Order of operations (the contract's, shared with the device kernels and the oracle): blocks of
// kGyroScanBlock samples, see gyro_scan.h.
void integrate_gyro(const double* timestamps_s, const double* gyro_xyz, size_t count, const double m[9],
                    double* quats_out /* count * 4 */);

}  // namespace rs
