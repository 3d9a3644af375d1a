"""Test-side reference of the gyro axis mapping as a 3x3 matrix (the rule of rssync_integrate_gyro_matrix,
DESIGN.md section 3.8), built on the CPU oracle without changing it.

map_gyro restates the rule with numpy's IEEE binary64 operations (no contraction): per output axis c,
w_c sums M[c][j] g_j over the j with M[c][j] != 0, the first kept term being the product and the others
added left to right; +0.0 when the row is zero.  The oracle's own integration with no orientation string
then computes a_c = (1.0 * w_c) * dt, and 1.0 * x == x for every binary64 x (signed zeros and NaNs
included), so integrate_gyro(ts, g, M) is the matrix integration under the contract's blocked order."""
import numpy as np


def map_gyro(matrix, gyro_xyz):
    """w = M g per sample under the zero-coefficient rule; rejects what the library rejects"""
    m = np.asarray(matrix, dtype=np.float64)
    if m.shape != (3, 3):
        raise ValueError(f"rotation must be 3x3, got shape {m.shape}")
    if not np.all(np.isfinite(m)):
        raise ValueError("rotation matrix with a non-finite entry")
    g = np.asarray(gyro_xyz, dtype=np.float64).reshape(-1, 3)
    w = np.zeros_like(g)
    for c in range(3):
        kept = False
        for j in range(3):
            if m[c, j] != 0.0:
                t = m[c, j] * g[:, j]
                w[:, c] = w[:, c] + t if kept else t
                kept = True
    return w


def integrate_gyro(oracle_loader, timestamps_s, gyro_xyz, matrix):
    """optdata_fill_gyro with the axis mapping `matrix`, on the oracle"""
    return oracle_loader.integrate_gyro(timestamps_s, map_gyro(matrix, gyro_xyz))


def rotation_search(oracle_loader, problem, timestamps_s, gyro_xyz, rotations, initial, fb, fe, step, radius):
    """the loop the rotation search stands for, on an OracleProblem: per matrix integrate, ingest through the
    variable-rate SetGyroQuaternions (timestamps truncated to integer microseconds), PreSync"""
    ts = np.ascontiguousarray(timestamps_s, dtype=np.float64)
    ts_us = (ts * 1000000).astype(np.int64)  # core_testcode.cpp:47-50 (truncation)
    out = []
    for r in rotations:
        problem.SetGyroQuaternions(ts_us, integrate_gyro(oracle_loader, ts, gyro_xyz, r), len(ts_us))
        out.append(problem.PreSync(initial, fb, fe, step, radius))
    return np.array([c for c, _ in out]), np.array([d for _, d in out])
