"""Windowed searches (rssync_readout_search_windows / rssync_rotation_search_windows, reached through
SyncProblem.readout_search_windows / rotation_search_windows).  Entry [j, w] is compared bit for bit with
the composed calls it stands for: PreSync over window w at call number call_nos[j W + w] on a problem
ingested at readout j, or after integrate_gyro(rotation=M_j) -> SetGyroQuaternions.  Plus W = 1 against
the single-window searches, the counter, side effects, errors, the recovery experiment through the engine
and several GPUs."""
import itertools

import numpy as np
import pytest

import plain_reference as ref
from conftest import workload
from test_gpu_readout_replicas import RAGGED_BASE, Source, _panic_frame
from test_gpu_readout_search import Frames, _problem, _state
from test_gpu_rotation_search import _rotations, _small
from test_readout_estimate import INITIAL, RADIUS, RECOVERY_TOL, SEEDS, STEP
from test_search_windows import (DRIFT, ROTATION_TOL_DEG, WINDOWS_TOL, recovery_scene, windows_of)
from test_gyro_rotation import RECOVERY_CASES, estimate_tilt_deg

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

N_GPUS = torch.cuda.device_count() if torch.cuda.is_available() else 0
# the engine's margin over the oracle in tests/test_readout_estimate.py: RECOVERY_TOL over its largest
# oracle error (0.23 ms)
ENGINE_MARGIN = RECOVERY_TOL - 0.00023


def _windows(s):
    """overlapping windows, an empty one, different lengths, pixel frames, row-fraction frames and one
    window mixing both"""
    p0, pe = s.pix.fb, s.pix.fe
    r0, re = s.rows.fb, s.rows.fe
    fb = [p0, p0 + 20, p0 + 290, r0 + 10, pe - 15, p0 + 5]
    fe = [p0 + 60, p0 + 50, p0 + 290, re, r0 + 12, p0 + 6]
    return np.array(fb, dtype=np.int64), np.array(fe, dtype=np.int64)


def _composed_readout(rsb, s, readouts, fb, fe, calls, simplified):
    """(costs, delays, curves) of fresh problems ingested at each readout, PreSync per window"""
    delays = rsb.presync_delays(INITIAL, STEP, RADIUS)
    n, W = len(readouts), len(fb)
    c, d, cv = np.empty((n, W)), np.empty((n, W)), np.empty((n, W, delays.size))
    for j, r in enumerate(readouts):
        q = s.ingest(_problem(rsb, s.w, simplified), r)
        for k in range(W):
            call = int(calls[j * W + k])
            cv[j, k] = q.presync_grid(int(fb[k]), int(fe[k]), delays, call_no=call)
            q.set_rng(100, call)
            c[j, k], d[j, k] = q.PreSync(INITIAL, int(fb[k]), int(fe[k]), STEP, RADIUS)
    return c, d, cv


def _equal(a, b):
    assert len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))


# ---- 1. readout form == re-ingested problems ------------------------------------------------------------
@pytest.mark.parametrize("simplified", [False, True], ids=["full", "simplified"])
def test_readout_windows_equal_reingest(rsb, synth_mod, simplified):
    s = Source(rsb, synth_mod, simplified)
    fb, fe = _windows(s)
    R = synth_mod.READOUT
    readouts = np.array([0.0, R, 1.7 * R])
    s.p.set_rng(100, 5)
    out = s.p.readout_search_windows(readouts, INITIAL, fb, fe, STEP, RADIUS, curves=True)
    n, W = len(readouts), len(fb)
    assert s.p.call_counter() == 5 + n * W
    assert out[0].shape == (n, W) and out[2].shape[:2] == (n, W)
    _equal(out, _composed_readout(rsb, s, readouts, fb, fe, 5 + np.arange(n * W), simplified))
    assert np.all(out[0][:, 2] == 0.0)  # the empty window
    # explicit call numbers, in any order
    calls = np.random.default_rng(1).permutation(n * W).astype(np.uint64) + 40
    out = s.p.readout_search_windows(readouts, INITIAL, fb, fe, STEP, RADIUS, call_nos=calls, curves=True)
    _equal(out, _composed_readout(rsb, s, readouts, fb, fe, calls, simplified))


# ---- 2. rotation form == the call sequence; strings through matrices ------------------------------------
def _rot_windows(fb0):
    return np.array([fb0, fb0 + 6, fb0 + 30, fb0 + 2], dtype=np.int64), np.array([fb0 + 12, fb0 + 24, fb0 + 30,
                                                                                     fb0 + 3], dtype=np.int64)


@pytest.mark.parametrize("simplified", [False, True], ids=["full", "simplified"])
def test_rotation_windows_equal_call_sequence(rsb, simplified):
    w, ts, fb0, _ = _small()
    fb, fe = _rot_windows(fb0)
    rots = _rotations(rsb, 3, 3)
    n, W = rots.shape[0], len(fb)
    g = rsb.SyncProblem(seed=100).load(w, bulk=True)
    g.set_loss_mode(simplified)
    table = g.frame_table().tobytes()
    g.set_rng(100, 3)
    cost, delay, curves = g.rotation_search_windows(ts, w.omega, rots, 0.0, fb, fe, 0.004, 0.06, curves=True)
    assert g.call_counter() == 3 + n * W and g.frame_table().tobytes() == table
    seq = rsb.SyncProblem(seed=100).load(w, bulk=True)
    seq.set_loss_mode(simplified)
    ts_us = (ts * 1000000).astype(np.int64)
    delays = rsb.presync_delays(0.0, 0.004, 0.06)
    for j, m in enumerate(rots):
        seq.SetGyroQuaternions(ts_us, rsb.integrate_gyro(ts, w.omega, rotation=m), len(ts_us))
        for k in range(W):
            call = 3 + j * W + k
            seq.set_rng(100, call)
            assert seq.PreSync(0.0, int(fb[k]), int(fe[k]), 0.004, 0.06) == (cost[j, k], delay[j, k])
            assert np.array_equal(seq.presync_grid(int(fb[k]), int(fe[k]), delays, call_no=call), curves[j, k])
    # the problem holds the last variant's gyro
    assert np.array_equal(g.probe_gyro()[2], seq.probe_gyro()[2]) and g.probe_gyro()[:2] == seq.probe_gyro()[:2]


def test_orientation_strings_through_matrices(rsb, synth_mod):
    w, ts, fb0, fe0 = _small()
    strings = synth_mod.ORIENTATIONS[:12]
    a = rsb.SyncProblem(seed=100).load(w, bulk=True)
    b = rsb.SyncProblem(seed=100).load(w, bulk=True)
    ca, da = a.orientation_search(ts, w.omega, strings, 0.0, fb0, fe0, 0.004, 0.06, call_nos=np.arange(12) + 2)
    cb, db = b.rotation_search_windows(ts, w.omega, [rsb.orientation_matrix(x) for x in strings], 0.0, [fb0], [fe0],
                                       0.004, 0.06, call_nos=np.arange(12) + 2)
    assert np.array_equal(ca, cb[:, 0]) and np.array_equal(da, db[:, 0])
    assert np.array_equal(a.probe_gyro()[2], b.probe_gyro()[2])


# ---- 3. W = 1 == the single-window searches -------------------------------------------------------------
def test_one_window_equals_single_window_searches(rsb, synth_mod):
    s = Source(rsb, synth_mod)
    readouts = np.array([0.0, 0.006, 0.013])
    for call_nos in (None, np.array([9, 4, 7], dtype=np.uint64)):
        s.p.set_rng(100, 21)
        a = s.p.readout_search(readouts, INITIAL, s.fb, s.fe, STEP, RADIUS, call_nos=call_nos, curves=True)
        ca = s.p.call_counter()
        s.p.set_rng(100, 21)
        b = s.p.readout_search_windows(readouts, INITIAL, [s.fb], [s.fe], STEP, RADIUS, call_nos=call_nos,
                                       curves=True)
        assert s.p.call_counter() == ca
        _equal(a, [x[:, 0] for x in b])
    w, ts, fb, fe = _small()
    rots = _rotations(rsb, 4, 4)
    g = rsb.SyncProblem(seed=100).load(w, bulk=True)
    for call_nos in (None, np.array([3, 1, 8, 8, 2], dtype=np.uint64)):
        g.set_rng(100, 6)
        a = g.rotation_search(ts, w.omega, rots, 0.0, fb, fe, 0.004, 0.06, call_nos=call_nos, curves=True)
        ca = g.call_counter()
        g.set_rng(100, 6)
        b = g.rotation_search_windows(ts, w.omega, rots, 0.0, [fb], [fe], 0.004, 0.06, call_nos=call_nos, curves=True)
        assert g.call_counter() == ca
        _equal(a, [x[:, 0] for x in b])


# ---- 4, 5. counter and problem state --------------------------------------------------------------------
def test_counter_and_state(rsb, synth_mod):
    s = Source(rsb, synth_mod)
    fb, fe = _windows(s)
    p = s.p
    p.set_rng(100, 11)
    before = (_state(p), p.retime_table().tobytes())
    readouts = [0.004, 0.011]
    a = p.readout_search_windows(readouts, INITIAL, fb, fe, STEP, RADIUS)
    assert p.call_counter() == 11 + 2 * len(fb)
    b = p.readout_search_windows(readouts, INITIAL, fb, fe, STEP, RADIUS, call_nos=11 + np.arange(2 * len(fb)))
    assert p.call_counter() == 11 + 2 * len(fb)
    _equal(a, b)
    assert (_state(p), p.retime_table().tobytes()) == before
    for r, f in (([], fb), (readouts, [])):
        c, d = p.readout_search_windows(r, INITIAL, f, f, STEP, RADIUS)
        assert c.shape == d.shape == (len(r), len(f))
    assert p.call_counter() == 11 + 2 * len(fb)
    st = p.stats()
    # the statistics are those of the last candidate's grid: every listed frame (overlaps counted again)
    listed = sum(int(np.count_nonzero((p.frame_table()["id"] >= b_) & (p.frame_table()["id"] < e_)))
                 for b_, e_ in zip(fb, fe))
    assert st["last_grid_tasks"] == listed * rsb.presync_delays(INITIAL, STEP, RADIUS).size
    # the rotation form: counter, and nothing done for no windows
    w, ts, fb0, _ = _small()
    rfb, rfe = _rot_windows(fb0)
    g = rsb.SyncProblem(seed=100).load(w, bulk=True)
    g.set_rng(100, 2)
    g.flush()
    rec = g.probe_gyro()[2]
    rots = _rotations(rsb, 5, 2)
    c, _ = g.rotation_search_windows(ts, w.omega, rots, 0.0, [], [], 0.004, 0.06)
    assert c.shape == (3, 0) and g.call_counter() == 2 and np.array_equal(g.probe_gyro()[2], rec)
    g.rotation_search_windows(ts, w.omega, rots, 0.0, rfb, rfe, 0.004, 0.06)
    assert g.call_counter() == 2 + 3 * len(rfb)
    g.rotation_search_windows(ts, w.omega, rots, 0.0, rfb, rfe, 0.004, 0.06, call_nos=np.zeros(3 * len(rfb)))
    assert g.call_counter() == 2 + 3 * len(rfb)


# ---- 6. errors ------------------------------------------------------------------------------------------
def _raises(rsb, fn, code, text=None):
    with pytest.raises(rsb.RsSyncError) as e:
        fn()
    assert e.value.code == code, e.value.message
    if text is not None:
        assert text in e.value.message, e.value.message
    return e.value.message


def test_readout_errors(rsb, synth_mod):
    s = Source(rsb, synth_mod)
    p = s.p
    w = s.w
    k = 9
    fid = 10 ** 6  # a rays frame: no row fractions
    p.SetTrackResult(fid, w.ts_a[k], w.ts_b[k], w.rays_a[k], w.rays_b[k], w.n_rays)
    p.SetTrackResult(fid + 1, w.ts_a[k], w.ts_b[k], w.rays_a[k], w.rays_b[k], w.n_rays)
    p.set_rng(100, 4)
    before = (_state(p), p.call_counter())
    fb, fe = np.array([s.pix.fb, fid - 5]), np.array([s.pix.fb + 30, fid + 2])
    _raises(rsb, lambda: p.readout_search_windows([0.01, 0.02], INITIAL, fb, fe, STEP, RADIUS), rsb.E_STATE,
            f"frame {fid} ")
    for bad in (np.nan, np.inf):
        _raises(rsb, lambda: p.readout_search_windows([0.01, bad], INITIAL, fb[:1], fe[:1], STEP, RADIUS),
                rsb.E_INVALID)
    with pytest.raises(ValueError):
        p.readout_search_windows([0.01], INITIAL, fb, fe[:1], STEP, RADIUS)
    with pytest.raises(ValueError):
        p.readout_search_windows([0.01], INITIAL, fb, fe, STEP, RADIUS, call_nos=[1])
    # the C entry point: negative counts, n W overflowing int, null buffers
    r = np.array([0.01])
    c, d = np.empty(2), np.empty(2)
    fbp, fep = fb.ctypes.data_as(rsb.c_i64_p), fe.ctypes.data_as(rsb.c_i64_p)
    dp = rsb.c_double_p
    call = p.L.rssync_readout_search_windows
    for n, W, a, b_, oc in ((-1, 1, fbp, fep, c), (1, -1, fbp, fep, c), (1 << 16, 1 << 16, fbp, fep, c),
                            (1, 2, None, fep, c), (1, 2, fbp, None, c), (1, 2, fbp, fep, None)):
        assert call(p.h, r.ctypes.data_as(dp), n, W, a, b_, INITIAL, STEP, RADIUS, None,
                    None if oc is None else oc.ctypes.data_as(dp), d.ctypes.data_as(dp), None) == rsb.E_INVALID
    assert (_state(p), p.call_counter()) == before


def test_rotation_errors(rsb):
    w, ts, fb0, _ = _small()
    fb, fe = _rot_windows(fb0)
    g = rsb.SyncProblem(seed=100).load(w, bulk=True)
    g.set_rng(100, 7)
    g.flush()
    rec = g.probe_gyro()[2]
    rots = _rotations(rsb, 5, 3)
    bad = rots.copy()
    bad[2, 1, 1] = np.nan
    _raises(rsb, lambda: g.rotation_search_windows(ts, w.omega, bad, 0.0, fb, fe, 0.004, 0.06), rsb.E_INVALID,
            "rotation-search: matrix 2 has a non-finite entry")
    m = rots.ravel().copy()
    c, d = np.empty(16), np.empty(16)
    dp = rsb.c_double_p
    fbp, fep = fb.ctypes.data_as(rsb.c_i64_p), fe.ctypes.data_as(rsb.c_i64_p)
    call = g.L.rssync_rotation_search_windows
    for n, W, mat, a, b_ in ((-1, 1, m, fbp, fep), (1, -1, m, fbp, fep), (1 << 16, 1 << 16, m, fbp, fep),
                             (2, 2, None, fbp, fep), (2, 2, m, None, fep), (2, 2, m, fbp, None)):
        assert call(g.h, ts.ctypes.data_as(dp), w.omega.ctypes.data_as(dp), ts.shape[0],
                    None if mat is None else mat.ctypes.data_as(dp), n, W, a, b_, 0.0, 0.004, 0.06, None,
                    c.ctypes.data_as(dp), d.ctypes.data_as(dp), None) == rsb.E_INVALID
    assert g.call_counter() == 7 and np.array_equal(g.probe_gyro()[2], rec)


def test_nonfinite_grid_reported_as_the_composed_calls(rsb, synth_mod):
    """a frame whose first estimator draw at call c_star is a pair of equal rays panics ("non-finite r") at
    every readout; placed in the second window of the second readout, the search fails as the composed
    calls do, and the same calls without c_star succeed"""
    w = workload("small")
    n, c_star = w.n_rays, 977
    fr, pair = _panic_frame(w, c_star, n)
    rest = Frames(w, rows=range(1, w.n_frames))
    D = rsb.presync_delays(0.0, 0.005, 0.02).size
    clean = (c for c in itertools.count() if c != c_star and all(
        {x, y} != set(pair) for d in range(D) for x, y in ref.draws(ref.rng_task_key(100, 1, c, d, fr.fb), 20, n)))
    calls = np.array(list(itertools.islice(clean, 6)), dtype=np.uint64)
    p = _problem(rsb, w)
    for f in (fr, rest):
        f.ingest(p, synth_mod, synth_mod.READOUT)
    fb, fe = np.array([fr.fb + 1, fr.fb]), np.array([fr.fb + 20, fr.fb + 20])
    args = ([0.0, 0.01, 0.02], 0.0, fb, fe, 0.005, 0.02)
    costs, _ = p.readout_search_windows(*args, call_nos=calls)
    assert np.isfinite(costs).all()
    bad = calls.copy()
    bad[1 * 2 + 1] = c_star
    msg = _raises(rsb, lambda: p.readout_search_windows(*args, call_nos=bad), rsb.E_NONFINITE)
    q = _problem(rsb, w)
    for f in (fr, rest):
        f.ingest(q, synth_mod, 0.01)
    q.set_rng(100, c_star)
    assert msg == _raises(rsb, lambda: q.PreSync(0.0, int(fb[1]), int(fe[1]), 0.005, 0.02), rsb.E_NONFINITE)
    assert msg == "pre-sync: non-finite r"


# ---- 7. recovery through the engine ---------------------------------------------------------------------
@pytest.mark.parametrize("drift", [None, DRIFT], ids=["constant", "drift"])
@pytest.mark.parametrize("seed", SEEDS)
def test_readout_recovery(rsb, synth_mod, seed, drift):
    from test_readout_estimate import READOUTS
    w = workload("C1", seed=seed, drift=drift)
    fr = Frames(w)
    p = fr.ingest(_problem(rsb, w), synth_mod, synth_mod.READOUT, device=True)
    fb, fe = windows_of(w)
    costs, _ = p.readout_search_windows(READOUTS, INITIAL, fb, fe, STEP, RADIUS)
    v = rsb.estimate_readout(READOUTS, costs.sum(axis=1))
    assert abs(v - synth_mod.READOUT) <= WINDOWS_TOL + ENGINE_MARGIN, (seed, drift, v)


@pytest.mark.parametrize("seed,axis,true_deg", RECOVERY_CASES)
def test_rotation_recovery(rsb, seed, axis, true_deg):
    w, ts, gyro, _ = recovery_scene(seed, axis, true_deg)
    fb, fe = windows_of(w)
    g = rsb.SyncProblem(seed=100).load(w, bulk=True)
    est = estimate_tilt_deg(
        lambda rots: g.rotation_search_windows(ts, gyro, rots, INITIAL, fb, fe, STEP, RADIUS)[0].sum(axis=1), axis)
    assert abs(est - true_deg) <= ROTATION_TOL_DEG, (seed, axis, true_deg, est)


# ---- 8. several GPUs ------------------------------------------------------------------------------------
@pytest.mark.skipif(N_GPUS < 2, reason="needs 2 GPUs")
def test_multi_device_equals_one_device(rsb, synth_mod):
    devices = list(range(min(N_GPUS, 4)))
    s = Source(rsb, synth_mod)
    multi = s.ingest(_problem(rsb, s.w, devices=devices), synth_mod.READOUT)
    fb, fe = _windows(s)
    readouts = np.linspace(0.0, 0.02, 2 * len(devices) + 1)
    res = []
    for p in (s.p, multi):  # the first windowed search after the ingest sends the row fractions
        p.set_rng(100, 3)
        out = p.readout_search_windows(readouts, INITIAL, fb, fe, STEP, RADIUS, curves=True)
        st = p.stats()
        res.append((out, p.call_counter(), st["last_grid_tasks"], st["last_grid_exact_tasks"]))
    _equal(res[0][0], res[1][0])
    assert res[0][1:] == res[1][1:]
    # an error: a frame without row fractions in the second window, on both
    for p in (s.p, multi):
        p.SetTrackResult(RAGGED_BASE + 5, s.w.ts_a[0], s.w.ts_b[0], s.w.rays_a[0], s.w.rays_b[0], s.w.n_rays)
    errs = [_raises(rsb, lambda: p.readout_search_windows(readouts, INITIAL, fb, fe, STEP, RADIUS), rsb.E_STATE)
            for p in (s.p, multi)]
    assert errs[0] == errs[1] and s.p.call_counter() == multi.call_counter()
    # the rotation form
    w, ts, fb0, _ = _small()
    rfb, rfe = _rot_windows(fb0)
    rots = _rotations(rsb, 6, 2 * len(devices))
    res = []
    for devs in (None, devices):
        g = rsb.SyncProblem(seed=100, devices=devs).load(w, bulk=True)
        g.set_rng(100, 4)
        out = g.rotation_search_windows(ts, w.omega, rots, 0.0, rfb, rfe, 0.004, 0.06, curves=True)
        st = g.stats()
        res.append((out, g.call_counter(), st["last_grid_tasks"], st["last_grid_exact_tasks"], g.probe_gyro()[2]))
    _equal(res[0][0], res[1][0])
    assert res[0][1:4] == res[1][1:4] and np.array_equal(res[0][4], res[1][4])
