"""The windowed searches (rssync_readout_search_windows / rssync_rotation_search_windows) on the CPU oracle:
the recovery experiments of tests/test_readout_estimate.py and tests/test_gyro_rotation.py with the cost of a
candidate summed over several syncpoint-sized frame windows, each with its own delay argmin, and the
symbols of the two entry points.

Every window's PreSync uses the RNG call number the windowed search gives a fresh problem: candidate j,
window w of W gets j * W + w (the rotation sweep's fine candidates continue where the coarse ones stop).
The largest error measured here pins the tolerances of the GPU recovery test
(tests/test_gpu_search_windows.py), which runs the same settings through the engine."""
import importlib
import os

import numpy as np
import pytest

import rotation_reference as rref
from conftest import workload
from test_abi import declared_symbols
from test_gyro_rotation import RECOVERY_CASES, estimate_tilt_deg, recovery_scene
from test_readout_estimate import INITIAL, RADIUS, READOUTS, SEEDS, STEP

# five 60-frame windows over C1's 300 frames
N_WINDOWS, WINDOW = 5, 60
# the delay drifts along the clip (2 ms/s, exaggerated so that a 5 s clip stands in for a long one)
DRIFT = (0.032, 0.042)
# |vertex - synth.READOUT| of the summed costs on the oracle, seeds 1, 2, 3: 0.29, 0.12, 0.16 ms with a
# constant delay and 0.27, 0.12, 0.32 ms with DRIFT.  For comparison, one 300-frame window
# (test_readout_estimate.retimed_minima) gives 0.23, 0.16, 0.05 ms with a constant delay and 0.07, 0.34,
# 0.43 ms with DRIFT; a single 60-frame window on its own is off by up to 2.1 ms.  The engine's rays differ
# from the host's by the rounding of tan / cos, hence some margin (as RECOVERY_TOL has over its errors).
WINDOWS_TOL = 0.0004
# |estimate - truth| of the mount tilt with the summed costs on the oracle, the cases of RECOVERY_CASES:
# 0.07, 0.03 and 0.58 degrees (the single-window sweep: 0.03, 0.39 and 0.68); the tolerance is
# RECOVERY_TOL_DEG's
ROTATION_TOL_DEG = 1.0


def _pkg():
    return importlib.import_module("rs-sync_b200")


def windows_of(w, n=N_WINDOWS, length=WINDOW):
    """n consecutive windows of `length` frames from w's first frame"""
    fb = int(w.frame_ids[0]) + length * np.arange(n, dtype=np.int64)
    return fb, fb + length


def retimed_window_minima(oracle_loader, w, readouts, synth_mod, fb, fe):
    """(n, W) PreSync minima on the oracle, rays re-timed on the host at each readout (as
    test_readout_estimate.retimed_minima), window w of candidate j keyed by call number j W + w"""
    delays = oracle_loader.presync_delays(INITIAL, STEP, RADIUS)
    tf_a = (w.frame_ids / w.fps)[:, None]
    tf_b = ((w.frame_ids + 1) / w.fps)[:, None]
    qa, qb = w.px_a[..., 1] / synth_mod.HEIGHT, w.px_b[..., 1] / synth_mod.HEIGHT
    W = len(fb)
    out = np.empty((len(readouts), W))
    for j, r in enumerate(readouts):
        o = oracle_loader.OracleProblem(threads=os.cpu_count() or 1, seed=100)
        o.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
        ts_a, ts_b = tf_a + r * qa, tf_b + r * qb
        for i, fid in enumerate(w.frame_ids):
            o.SetTrackResult(int(fid), ts_a[i], ts_b[i], w.rays_a[i], w.rays_b[i], w.n_rays)
        for k in range(W):
            out[j, k] = float(np.min(o.presync_grid(int(fb[k]), int(fe[k]), delays, call_no=j * W + k)))
    return out


def rotation_window_minima(oracle_loader, o, ts, gyro, rotations, fb, fe):
    """(n, W) PreSync minima on the oracle per rotation and window, in the windowed search's order: the
    problem's counter keys them"""
    ts_us = (np.ascontiguousarray(ts, dtype=np.float64) * 1000000).astype(np.int64)
    out = np.empty((len(rotations), len(fb)))
    for j, r in enumerate(rotations):
        o.SetGyroQuaternions(ts_us, rref.integrate_gyro(oracle_loader, ts, gyro, r), len(ts_us))
        for k in range(len(fb)):
            out[j, k] = o.PreSync(INITIAL, int(fb[k]), int(fe[k]), STEP, RADIUS)[0]
    return out


@pytest.mark.parametrize("drift", [None, DRIFT], ids=["constant", "drift"])
@pytest.mark.parametrize("seed", SEEDS)
def test_readout_recovery_across_windows(oracle_loader, synth_mod, seed, drift):
    w = workload("C1", seed=seed, drift=drift)
    fb, fe = windows_of(w)
    costs = retimed_window_minima(oracle_loader, w, READOUTS, synth_mod, fb, fe)
    v = _pkg().estimate_readout(READOUTS, costs.sum(axis=1))
    assert abs(v - synth_mod.READOUT) <= WINDOWS_TOL, (seed, drift, v)


@pytest.mark.parametrize("seed,axis,true_deg", RECOVERY_CASES)
def test_rotation_recovery_across_windows(oracle_loader, seed, axis, true_deg):
    w, ts, gyro, _ = recovery_scene(seed, axis, true_deg)
    fb, fe = windows_of(w)
    o = oracle_loader.OracleProblem(threads=os.cpu_count() or 1, seed=100).load(w)
    est = estimate_tilt_deg(
        lambda rots: rotation_window_minima(oracle_loader, o, ts, gyro, rots, fb, fe).sum(axis=1), axis)
    assert abs(est - true_deg) <= ROTATION_TOL_DEG, (seed, axis, true_deg, est)


def test_symbols_exported_and_declared(rsb):
    lib = rsb.load_library()
    for name in ("rssync_readout_search_windows", "rssync_rotation_search_windows"):
        assert name in declared_symbols() and name in rsb.C_ABI_SYMBOLS, name
        assert hasattr(lib, name), name
