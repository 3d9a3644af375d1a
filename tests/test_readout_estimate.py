"""estimate_readout (the vertex of a least-squares parabola through (readout, PreSync minimum) points) and
the readout-recovery experiment on the CPU oracle.

The recovery experiment re-times synthetic C1 scenes, generated with the readout synth.READOUT, at
candidate readouts 0 .. 22 ms on the host (ts = frame_ts + r * (y / HEIGHT), the pixel ingest's
expression; the rays do not depend on the readout) and takes the minimum of one PreSync grid per
candidate, with the RNG call numbers rssync_readout_search gives a fresh problem (0, 1, ...).  The
largest error it measures pins the tolerance of the GPU recovery test (tests/test_gpu_readout_search.py),
which runs the same settings through the engine."""
import importlib
import os

import numpy as np
import pytest

from conftest import workload

# the recovery settings, shared with the GPU test
READOUTS = np.arange(0.0, 0.0221, 0.002)  # 0, 2, ..., 22 ms
INITIAL, STEP, RADIUS = 0.037, 0.0005, 0.012
SEEDS = (1, 2, 3)
# |vertex - synth.READOUT| the oracle gives on these scenes: 0.23, 0.16 and 0.05 ms for seeds 1, 2, 3; the
# engine's rays differ from the host's by the rounding of tan / cos, hence some margin
RECOVERY_TOL = 0.0003


def _pkg():
    return importlib.import_module("rs-sync_b200")


def test_exact_parabolas():
    est = _pkg().estimate_readout
    for vertex, a, c0 in [(0.011, 3.0e6, 120.0), (0.0005, 1.0, 0.0), (0.0173, 5.0e4, -7.0), (0.02, 2.0e8, 1e6)]:
        r = np.arange(0.0, 0.0221, 0.002)
        c = a * (r - vertex) ** 2 + c0
        assert est(r, c) == pytest.approx(vertex, abs=1e-12)
    # unsorted candidates, exactly three of them
    r = np.array([0.004, 0.0, 0.002])
    assert est(r, (r - 0.0015) ** 2) == pytest.approx(0.0015, abs=1e-14)


def test_rejections():
    est = _pkg().estimate_readout
    r = np.arange(0.0, 0.0221, 0.002)
    with pytest.raises(ValueError, match="not convex"):
        est(r, -(r - 0.011) ** 2)
    with pytest.raises(ValueError, match="not convex"):
        est(r, 2.0 * r + 1.0)  # a straight line
    with pytest.raises(ValueError, match="outside"):
        est(r, (r - 0.03) ** 2)
    with pytest.raises(ValueError, match="outside"):
        est(r, (r + 0.001) ** 2)
    with pytest.raises(ValueError, match="3 distinct"):
        est([0.01, 0.01, 0.02], [1.0, 1.0, 2.0])
    with pytest.raises(ValueError, match="costs"):
        est(r, r[:-1])
    with pytest.raises(ValueError, match="finite"):
        est(r, np.where(r > 0.01, np.nan, r))


def retimed_minima(oracle_loader, w, readouts, synth_mod, simplified=False):
    """PreSync minimum per candidate readout on the oracle, rays re-timed on the host"""
    delays = oracle_loader.presync_delays(INITIAL, STEP, RADIUS)
    tf_a = (w.frame_ids / w.fps)[:, None]
    tf_b = ((w.frame_ids + 1) / w.fps)[:, None]
    qa, qb = w.px_a[..., 1] / synth_mod.HEIGHT, w.px_b[..., 1] / synth_mod.HEIGHT
    out = []
    for j, r in enumerate(readouts):
        o = oracle_loader.OracleProblem(threads=os.cpu_count() or 1, seed=100)
        o.set_loss_mode(simplified)
        o.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
        ts_a, ts_b = tf_a + r * qa, tf_b + r * qb
        for i, fid in enumerate(w.frame_ids):
            o.SetTrackResult(int(fid), ts_a[i], ts_b[i], w.rays_a[i], w.rays_b[i], w.n_rays)
        fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
        out.append(float(np.min(o.presync_grid(fb, fe, delays, call_no=j))))
    return np.array(out)


@pytest.mark.parametrize("seed", SEEDS)
def test_recovery_on_the_oracle(oracle_loader, synth_mod, seed):
    w = workload("C1", seed=seed)
    costs = retimed_minima(oracle_loader, w, READOUTS, synth_mod)
    v = _pkg().estimate_readout(READOUTS, costs)
    assert abs(v - synth_mod.READOUT) <= RECOVERY_TOL, (seed, v, costs)
