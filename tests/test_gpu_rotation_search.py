"""Rotation search (rssync_rotation_search, reached through SyncProblem.rotation_search): PreSync under
arbitrary 3x3 gyro axis mappings, run on the device by the orientation search's pipeline.  Checked bit for
bit against the orientation search (the 48 signed permutation matrices), against the caller's sequence of
calls (integrate_gyro(rotation=) -> SetGyroQuaternions -> PreSync / presync_grid), and against the
oracle's loop of host calls; plus counter handling, side effects, rejections, the recovery of a known
mount tilt and two GPUs."""
import ctypes as C

import numpy as np
import pytest

import rotation_reference as ref
from conftest import rel_err, workload
from test_gyro_rotation import (INITIAL, RADIUS, RECOVERY_CASES, RECOVERY_TOL_DEG, STEP, estimate_tilt_deg,
                                recovery_scene)

pytestmark = pytest.mark.gpu

TOL = 1e-9  # loss-curve values against the oracle, as tests/test_gpu_parity.py


def _small():
    w = workload("small")
    ts = w.gyro_t0 + np.arange(w.quats.shape[0]) / w.gyro_rate
    fb = int(w.frame_ids[0])
    return w, ts, fb, fb + 24


def _rotations(rsb, seed, n):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        axis = rng.normal(size=3)
        axis /= np.linalg.norm(axis)
        th = rng.uniform(-0.6, 0.6)
        k = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
        out.append(np.eye(3) + np.sin(th) * k + (1 - np.cos(th)) * (k @ k))  # Rodrigues
    out.append(rsb.rotations_about("y", [0.3])[0] @ rsb.orientation_matrix("yXz"))
    return np.array(out)


def test_matrices_equal_strings(rsb, synth_mod):
    """the 48 signed permutation matrices give the orientation search's results, counter and gyro bit for bit"""
    w, ts, fb, fe = _small()
    assert ts.shape[0] > 3 * 512
    a = rsb.SyncProblem(seed=100).load(w, bulk=True)
    b = rsb.SyncProblem(seed=100).load(w, bulk=True)
    a.set_rng(100, 5)
    b.set_rng(100, 5)
    ca, da = a.orientation_search(ts, w.omega, synth_mod.ORIENTATIONS, 0.0, fb, fe, 0.004, 0.06)
    mats = [rsb.orientation_matrix(s) for s in synth_mod.ORIENTATIONS]
    cb, db = b.rotation_search(ts, w.omega, mats, 0.0, fb, fe, 0.004, 0.06)
    assert np.array_equal(ca, cb) and np.array_equal(da, db)
    assert a.call_counter() == b.call_counter() == 5 + 48
    assert np.array_equal(a.probe_gyro()[2], b.probe_gyro()[2])


@pytest.mark.parametrize("simplified", [False, True])
def test_search_equals_call_sequence_and_oracle(rsb, oracle_loader, simplified):
    w, ts, fb, fe = _small()
    rots = _rotations(rsb, 3, 5)
    n = rots.shape[0]
    g = rsb.SyncProblem(seed=100).load(w, bulk=True)
    g.set_loss_mode(simplified)
    table = g.frame_table().tobytes()
    g.set_rng(100, 3)
    cost, delay, curves = g.rotation_search(ts, w.omega, rots, 0.0, fb, fe, 0.004, 0.06, curves=True)
    assert g.call_counter() == 3 + n
    assert g.frame_table().tobytes() == table  # the tracks are untouched
    # the oracle's loop of host calls
    o = oracle_loader.OracleProblem(threads=8, seed=100).load(w)
    o.set_loss_mode(simplified)
    o.set_rng(100, 3)
    co, do = ref.rotation_search(oracle_loader, o, ts, w.omega, rots, 0.0, fb, fe, 0.004, 0.06)
    assert np.array_equal(delay, do) and rel_err(cost, co) <= TOL
    # the caller's sequence of calls on the engine, result j keyed by call number 3 + j
    seq = rsb.SyncProblem(seed=100).load(w, bulk=True)
    seq.set_loss_mode(simplified)
    ts_us = (ts * 1000000).astype(np.int64)
    delays = rsb.presync_delays(0.0, 0.004, 0.06)
    assert curves.shape == (n, delays.shape[0])
    for j, m in enumerate(rots):
        seq.SetGyroQuaternions(ts_us, rsb.integrate_gyro(ts, w.omega, rotation=m), len(ts_us))
        seq.set_rng(100, 3 + j)
        assert seq.PreSync(0.0, fb, fe, 0.004, 0.06) == (cost[j], delay[j])
        assert np.array_equal(seq.presync_grid(fb, fe, delays, call_no=3 + j), curves[j])
    # the problem holds the last variant's gyro
    assert np.array_equal(g.probe_gyro()[2], seq.probe_gyro()[2])
    assert g.probe_gyro()[:2] == seq.probe_gyro()[:2]


def test_explicit_call_numbers_and_empty_search(rsb):
    w, ts, fb, fe = _small()
    rots = _rotations(rsb, 4, 5)
    g = rsb.SyncProblem(seed=100).load(w, bulk=True)
    g.set_rng(100, 11)
    cost, delay = g.rotation_search(ts, w.omega, rots, 0.0, fb, fe, 0.004, 0.06)
    before = g.call_counter()
    sub = [4, 0, 2]
    cs, ds, cv = g.rotation_search(ts, w.omega, rots[sub], 0.0, fb, fe, 0.004, 0.06,
                                   call_nos=np.array([11 + k for k in sub], dtype=np.uint64), curves=True)
    assert np.array_equal(cs, cost[sub]) and np.array_equal(ds, delay[sub])
    assert g.call_counter() == before
    # the problem holds the subset's last variant's gyro (rots[2], call number 13)
    assert np.array_equal(cv[2], g.presync_grid(fb, fe, rsb.presync_delays(0.0, 0.004, 0.06), call_no=13))
    rec = g.probe_gyro()[2]
    for empty in ([], np.zeros((0, 3, 3))):
        c0, d0 = g.rotation_search(ts, w.omega, empty, 0.0, fb, fe, 0.004, 0.06)
        assert c0.shape == d0.shape == (0,)
    assert g.call_counter() == before and np.array_equal(g.probe_gyro()[2], rec)


def test_rejections(rsb):
    w, ts, fb, fe = _small()
    g = rsb.SyncProblem(seed=100).load(w, bulk=True)
    g.set_rng(100, 7)
    g.flush()
    rec = g.probe_gyro()[2]
    good = _rotations(rsb, 5, 3)

    def unchanged():
        assert g.call_counter() == 7
        assert np.array_equal(g.probe_gyro()[2], rec)

    for bad in (np.nan, np.inf):
        rots = good.copy()
        rots[2, 1, 0] = bad
        with pytest.raises(rsb.RsSyncError) as e:
            g.rotation_search(ts, w.omega, rots, 0.0, fb, fe, 0.004, 0.06)
        assert e.value.code == rsb.E_INVALID
        assert e.value.message == "rotation-search: matrix 2 has a non-finite entry"
        unchanged()
    # a null matrix array with n > 0
    cost, delay = np.empty(2), np.empty(2)
    ts64, om = np.ascontiguousarray(ts), np.ascontiguousarray(w.omega)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    rc = g.L.rssync_rotation_search(g.h, dp(ts64), dp(om), ts64.shape[0], None, 2, 0.0, fb, fe, 0.004, 0.06, None,
                                    dp(cost), dp(delay), None)
    assert rc == rsb.E_INVALID
    unchanged()
    # the orientation search's own checks, reached through the shared body
    cases = [
        ((ts[:1], w.omega[:1], 0.004, 0.06), rsb.E_INVALID, "set-gyro-quaternions: need at least 2 samples"),
        ((ts, w.omega, 0.0, 0.06), rsb.E_INVALID, "pre-sync: search_step must be > 0 and the search window finite"),
        ((ts, w.omega, 0.004, np.inf), rsb.E_INVALID,
         "pre-sync: search_step must be > 0 and the search window finite"),
    ]
    for (t, om_, step, radius), code, msg in cases:
        with pytest.raises(rsb.RsSyncError) as e:
            g.rotation_search(t, om_, good, 0.0, fb, fe, step, radius)
        assert e.value.code == code and e.value.message == msg
        unchanged()
    swapped = ts.copy()
    swapped[[10, 11]] = swapped[[11, 10]]
    with pytest.raises(rsb.RsSyncError) as e:
        g.rotation_search(swapped, w.omega, good, 0.0, fb, fe, 0.004, 0.06)
    assert e.value.code == rsb.E_ORDER and e.value.message.startswith("set-gyro-quaternions:  timestamps out of order")
    unchanged()
    with pytest.raises(ValueError, match="3x3"):
        g.rotation_search(ts, w.omega, np.zeros((2, 3)), 0.0, fb, fe, 0.004, 0.06)
    with pytest.raises(ValueError, match="call numbers"):
        g.rotation_search(ts, w.omega, good, 0.0, fb, fe, 0.004, 0.06, call_nos=[1])
    unchanged()


@pytest.mark.parametrize("seed,axis,true_deg", RECOVERY_CASES)
def test_recovery(rsb, seed, axis, true_deg):
    w, ts, gyro, (fb, fe) = recovery_scene(seed, axis, true_deg)
    p = rsb.SyncProblem(seed=100).load(w, bulk=True)
    est = estimate_tilt_deg(lambda rots: p.rotation_search(ts, gyro, rots, INITIAL, fb, fe, STEP, RADIUS)[0], axis)
    assert abs(est - true_deg) <= RECOVERY_TOL_DEG, (seed, axis, true_deg, est)
    # applying the estimate: the integrated gyro goes in through SetGyroQuaternions as usual
    r = rsb.rotations_about(axis, [np.deg2rad(est)])[0]
    p.SetGyroQuaternions((ts * 1000000).astype(np.int64), rsb.integrate_gyro(ts, gyro, rotation=r), len(ts))
    assert abs(p.PreSync(INITIAL, fb, fe, STEP, RADIUS)[1] - 0.037) <= 0.002


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_n_gpus() < 2, reason="needs 2 GPUs")
def test_two_devices(rsb):
    w, ts, fb, fe = _small()
    rots = _rotations(rsb, 6, 6)
    one = rsb.SyncProblem(seed=100).load(w, bulk=True)
    many = rsb.SyncProblem(seed=100, devices=[0, 1]).load(w, bulk=True)
    for p in (one, many):
        p.set_rng(100, 2)
    a = one.rotation_search(ts, w.omega, rots, 0.0, fb, fe, 0.004, 0.06, curves=True)
    b = many.rotation_search(ts, w.omega, rots, 0.0, fb, fe, 0.004, 0.06, curves=True)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    assert one.call_counter() == many.call_counter() == 2 + rots.shape[0]
    assert np.array_equal(one.probe_gyro()[2], many.probe_gyro()[2])
    for p in (one, many):
        p.set_rng(100, 20)
    assert one.PreSync(0.0, fb, fe, 0.004, 0.06) == many.PreSync(0.0, fb, fe, 0.004, 0.06)
    bad = rots.copy()
    bad[4, 0, 0] = np.nan
    with pytest.raises(rsb.RsSyncError) as e:
        many.rotation_search(ts, w.omega, bad, 0.0, fb, fe, 0.004, 0.06)
    assert e.value.message == "rotation-search: matrix 4 has a non-finite entry"
    assert many.call_counter() == 21
