"""The translation estimator on frames built to tie (tests/estimator_frames.py), against the CPU oracle
and its per-hypothesis trace: the product path (fp32 tournament, packed pairs, prior threshold, value
selects, exact settles) must return the exact binary64 estimator's M bit for bit, and an exact tie must
go to the earlier hypothesis (core_private.cpp:53, strict <).  Random frames practically never tie, so
the rest of the suite cannot tell a wrong tie-break from a right one.

Also: a finite row of norm < 1e-12 (a static ray pair) must not raise "non-finite numbers in P"."""
import numpy as np
import pytest

import estimator_frames as ef
import plain_reference as pr
from conftest import rel_err, workload
from test_estimator_ties import stream_of, threshold_cases, tie_cases

pytestmark = pytest.mark.gpu

TOL = 1e-9


def designed_frames(n, oracle_loader, grid_offsets=None):
    """families a (every tie placement), c (both variants), d; with grid_offsets, the 20-hypothesis
    frames are designed for those offset indices of a grid (one per frame, in turn)"""
    frames, k = [], 0

    def off():
        nonlocal k
        k += 1
        return 0 if grid_offsets is None else grid_offsets[(k - 1) % len(grid_offsets)]

    for t1, t2, iters in tie_cases(n):
        if grid_offsets is not None and iters == 200:
            continue
        frames.append(ef.mirror_frame(n, t1, t2, iters, stream_of(iters), offset=off(), fid0=1000 + 1000 * k,
                                      oracle_loader=oracle_loader))
    for zv in (False, True):
        for iters in ((20,) if grid_offsets is not None else (20, 200)):
            frames.append(ef.zero_frame(n, zv, t1=0 if n < 64 else 3, iters=iters, stream=stream_of(iters),
                                        offset=off(), fid0=20000 + 1000 * k, oracle_loader=oracle_loader))
    for iters in ((20,) if grid_offsets is not None else (20, 200)):
        frames.append(ef.repeated_frame(n, iters, stream_of(iters), offset=off(), fid0=40000 + 1000 * k))
    assert len({f.fid for f in frames}) == len(frames)
    return frames


def pair(rsb, oracle_loader, frames):
    g = ef.load_gyro(rsb.SyncProblem(seed=ef.SEED))
    for f in frames:
        f.load(g)
    return g, ef.oracle_problem(oracle_loader, frames, threads=8)


@pytest.mark.parametrize("n", ef.N_RAYS)
def test_probes_on_designed_frames(rsb, oracle_loader, n):
    """20 hypotheses (stream 1) and 200 (stream 3): product path == exact estimator == oracle == the
    trace's winner, M bits and k; on exact ties (families a, c) that is t1's M, not t2's"""
    frames = designed_frames(n, oracle_loader)
    g, o = pair(rsb, oracle_loader, frames)
    for f in frames:
        v, q, best = o.estimator_trace(f.fid, 0.0, f.iters, f.stream, f.call_no, f.offset)
        mo, ko = o.guess_motion(f.fid, 0.0, f.iters, f.stream, f.call_no, f.offset)
        assert np.array_equal(ef.bits(mo), ef.bits(v[best]))
        for mode in (0, 2):
            mg, kg, _ = g.probe_guess_motion_ex(f.fid, 0.0, f.iters, f.stream, f.call_no, f.offset, mode)
            assert np.array_equal(ef.bits(mg), ef.bits(mo)), (f.family, n, f.t1, f.t2, mode, mg, mo)
            assert kg == ko or (np.isnan(kg) and np.isnan(ko)), (f.family, n, mode, kg, ko)
        if f.family in ("a", "c", "c0"):
            assert best == f.t1 and q[f.t1] == q[f.t2]
            assert not np.array_equal(ef.bits(mg), ef.bits(v[f.t2]))


@pytest.mark.parametrize("n", [n for n in ef.N_RAYS if n >= 32])
def test_near_ties_across_the_margin(rsb, oracle_loader, n):
    """t2's rays rotated by eps: its quartile gap to t1 sweeps from far inside the fp32 band (the
    comparison must be settled in binary64) to far outside it (it must not be); the winner is the
    oracle's either way.  t1 is hypothesis 0 and every other hypothesis is far from both, so the
    settle is the designed one."""
    g = ef.load_gyro(rsb.SyncProblem(seed=ef.SEED))
    for iters in (20, 200):
        frames = ef.near_tie_sweep(n, iters, stream_of(iters), oracle_loader=oracle_loader)
        used = {}
        for f in frames:
            f.load(g)
            o = ef.oracle_problem(oracle_loader, [f])
            mo, ko = o.guess_motion(f.fid, 0.0, iters, f.stream, f.call_no, f.offset)
            mg, kg, u = g.probe_guess_motion_ex(f.fid, 0.0, iters, f.stream, f.call_no, f.offset, 0)
            assert np.array_equal(ef.bits(mg), ef.bits(mo)) and kg == ko, (n, iters, f.meta)
            gap = f.meta["gap"]
            if gap <= 0.05 * ef.K_MARGIN:
                assert u == 1, (n, iters, f.meta)
            if gap >= 2 * ef.K_MARGIN:
                assert u == 0, (n, iters, f.meta)
            used[f.meta["eps"]] = u
        eps = sorted(used, key=abs)
        assert used[eps[0]] == used[eps[1]] == 1 and used[eps[-1]] == used[eps[-2]] == 0
        assert set(used.values()) == {0, 1}


def _cell_bounds(o, frames, delays, call_no):
    """every (delay, frame) cell of the oracle against plain_reference.presync_cell's bound"""
    rec = o.spline()
    fc_all = {}
    for f in frames:
        c, fc, _ = o.presync_grid(f.fid, f.fid + 1, delays, call_no=call_no, frame_costs=True)
        fc_all[f.fid] = fc[:, 0]
        for di, delay in enumerate(delays):
            P = pr.rows(rec, ef.GYRO_T0, ef.GYRO_RATE, delay, f.ts_a, f.ts_b, f.rays_a, f.rays_b)
            key = pr.rng_task_key(ef.SEED, ef.STREAM_PRESYNC, call_no, di, f.fid)
            got = fc[di, 0]
            if not np.isfinite(got):
                continue
            cands = [(c, b) for c, b in pr.presync_cell(P, key) if np.isfinite(c)]
            assert pr.cell_ratio(got, cands) <= 1.0, (f.family, f.fid, di)
    return fc_all


@pytest.mark.parametrize("n_delays", [16, 5], ids=["staged-prior", "unstaged"])
@pytest.mark.parametrize("n", ef.N_RAYS)
def test_grid_on_designed_frames(rsb, oracle_loader, n, n_delays):
    """the PreSync grid over the designed frames: 16 consecutive delays (staged, the prior path active)
    and 5; each frame's tie falls on a different offset index, so on first and later tasks of a warp's
    group.  Costs and flags equal the oracle's; each frame's cells are within the plain reference's bound"""
    offsets = [0, 5, 2, 15, 7, 10, 3, 12, 1] if n_delays == 16 else [0, 4, 2, 1, 3]
    frames = designed_frames(n, oracle_loader, grid_offsets=offsets)
    g, o = pair(rsb, oracle_loader, frames)
    delays = np.linspace(-0.03, 0.045, n_delays)
    fb, fe = min(f.fid for f in frames), max(f.fid for f in frames) + 1
    cg, flg = g.presync_grid(fb, fe, delays, call_no=0, return_flags=True)
    co, _, flo = o.presync_grid(fb, fe, delays, call_no=0, frame_costs=True)
    assert np.array_equal(cg, co, equal_nan=True)
    assert flg == flo
    fc = _cell_bounds(o, frames, delays, 0)
    for f in frames:  # the engine's cells, one frame at a time, equal the oracle's
        cf, ff = g.presync_grid(f.fid, f.fid + 1, delays, call_no=0, return_flags=True)
        assert np.array_equal(cf, fc[f.fid], equal_nan=True), (f.family, f.fid)


@pytest.mark.parametrize("n", ef.N_RAYS)
def test_sync_on_designed_frames(rsb, oracle_loader, n):
    """Sync's initialisation (200 hypotheses, sync_init_kernel) on designed frames, one Sync per frame
    with the call number its tie was designed for"""
    frames = [ef.mirror_frame(n, t1, t2, 200, ef.STREAM_SYNCINIT, call_no=c, fid0=60000 + 1000 * c,
                              oracle_loader=oracle_loader)
              for c, (t1, t2) in enumerate([(31, 32), (193, 198)]) if n >= 32]
    frames.append(ef.zero_frame(n, False, t1=0 if n < 64 else 3, iters=200, stream=ef.STREAM_SYNCINIT,
                                call_no=2, fid0=70000, oracle_loader=oracle_loader))
    rep = ef.repeated_frame(n, 200, ef.STREAM_SYNCINIT, call_no=3, fid0=80000)
    if all(rep.meta["group"][a] != rep.meta["group"][b] for a, b in ef._draws(rep.fid, n, 3, 3, 0, 200)):
        frames.append(rep)  # (otherwise the zero hypothesis of two copies wins: M = 0, no loss to minimise)
    g, o = pair(rsb, oracle_loader, frames)
    fb = np.array([f.fid for f in frames], dtype=np.int64)
    cn = np.array([f.call_no for f in frames], dtype=np.uint64)
    ini = np.zeros(len(frames))
    cg, dg = g.sync_batch(ini, fb, fb + 1, 0.0, 0.1, call_nos=cn)
    co, do = o.sync_batch(ini, fb, fb + 1, 0.0, 0.1, call_nos=cn)
    assert rel_err(cg, co) <= TOL and np.max(np.abs(dg - do)) <= TOL * max(1.0, np.max(np.abs(do)))


@pytest.mark.parametrize("n", [n for n in ef.N_RAYS if n >= 32])
def test_rows_at_the_normalisation_threshold(rsb, oracle_loader, n):
    """rows of norm just below 1e-12, whose fp32 |row|^2 rounds to fp32(1e-24): the fp32 tournament must
    hand them to the exact estimator like any row safe_normalize leaves unscaled -- normalised, they
    move the winner by more than the margin (the builder's precondition)"""
    for iters, stream in threshold_cases(n):
        f = ef.threshold_rows_frame(n, iters, stream, oracle_loader=oracle_loader)
        g, o = pair(rsb, oracle_loader, [f])
        mo, ko = o.guess_motion(f.fid, 0.0, iters, stream, f.call_no, f.offset)
        for mode in (0, 2):
            mg, kg, _ = g.probe_guess_motion_ex(f.fid, 0.0, iters, stream, f.call_no, f.offset, mode)
            assert np.array_equal(ef.bits(mg), ef.bits(mo)) and kg == ko, (n, iters, mode, mg, mo)
        if iters == 20:
            delays = np.linspace(-0.03, 0.045, 16)
            cg, flg = g.presync_grid(f.fid, f.fid + 1, delays, return_flags=True)
            co, _, flo = o.presync_grid(f.fid, f.fid + 1, delays, frame_costs=True)
            assert np.array_equal(cg, co, equal_nan=True) and flg == flo


# ---- tiny finite rows ------------------------------------------------------------------------------
STEP, RADIUS = 0.005, 0.05


def _static_problems(rsb, oracle_loader, frames, w):
    g = rsb.SyncProblem(seed=ef.SEED).load(w)
    o = oracle_loader.OracleProblem(threads=4, seed=ef.SEED).load(w)
    for f in frames:
        f.load(g)
        f.load(o)
    return g, o


def _entry_points(p, w, fb, fe, oracle_loader=None):
    """PreSync, DebugPreSync, two PreSync windows and an orientation search, RNG call numbers fixed"""
    out = []
    p.set_rng(ef.SEED, 7)
    out.append(p.PreSync(0.0, fb, fe, STEP, RADIUS))
    p.set_rng(ef.SEED, 8)
    out.append(p.DebugPreSync(0.0, fb, fe, RADIUS, 21))
    mid = (fb + fe) // 2
    if oracle_loader is None:
        out.append(p.presync_windows(0.0, [fb, mid], [mid, fe], STEP, RADIUS, call_nos=[9, 10]))
    else:
        r = []
        for c, (b, e) in ((9, (fb, mid)), (10, (mid, fe))):
            p.set_rng(ef.SEED, c)
            r.append(p.PreSync(0.0, b, e, STEP, RADIUS))
        out.append((np.array([x[0] for x in r]), np.array([x[1] for x in r])))
    ts = w.gyro_t0 + np.arange(w.quats.shape[0]) / w.gyro_rate
    p.set_rng(ef.SEED, 11)
    if oracle_loader is None:
        out.append(p.orientation_search(ts, w.omega, ["XYZ", "yXz"], 0.0, fb, fe, STEP, RADIUS))
    else:
        out.append(oracle_loader.orientation_search(p, ts, w.omega, ["XYZ", "yXz"], 0.0, fb, fe, STEP, RADIUS))
    return out


def _assert_same(rg, ro):
    (cg, dg), (dgd, cgd), (wcg, wdg), (ocg, odg) = rg
    (co, do), (dod, cod), (wco, wdo), (oco, odo) = ro
    assert dg == do and rel_err(cg, co) <= TOL
    assert np.array_equal(dgd, dod) and rel_err(cgd, cod) <= TOL
    assert np.array_equal(wdg, wdo) and rel_err(wcg, wco) <= TOL
    assert np.array_equal(odg, odo) and rel_err(ocg, oco) <= TOL


def test_static_pair_is_not_a_panic(rsb, oracle_loader):
    """a frame with one static ray pair (b = a, ts_b = ts_a): its row is finite, of norm < 1e-12, and
    goes to the exact estimator; the entry points return the oracle's results, no error.  Variants: the
    static pair avoided by one designed task's draws, and drawn (its unnormalised hypothesis wins)"""
    w = workload("tiny", first_frame=200)
    frames = [ef.with_static_pair(w, 2, 0, drawn=False, call_no=7, offset=3),
              ef.with_static_pair(w, 5, 0, drawn=True, call_no=7, offset=4),
              ef.with_static_pair(w, 9, 11)]
    g, o = _static_problems(rsb, oracle_loader, frames, w)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    _assert_same(_entry_points(g, w, fb, fe), _entry_points(o, w, fb, fe, oracle_loader))
    for f in frames:  # the designed tasks, probed
        mo, ko = o.guess_motion(f.fid, 0.0, 20, f.stream, f.call_no, f.offset)
        mg, kg, used = g.probe_guess_motion_ex(f.fid, 0.0, 20, f.stream, f.call_no, f.offset, 0)
        assert np.array_equal(ef.bits(mg), ef.bits(mo)) and kg == ko and used == 1


def test_all_static_frame(rsb, oracle_loader):
    """every ray pair of a frame static: both sides agree, whether that is a result or an error"""
    w = workload("tiny", first_frame=200)
    f = ef.all_static(w, 0)
    g, o = _static_problems(rsb, oracle_loader, [f], w)
    fb, fe = int(w.frame_ids[0]), f.fid + 1
    try:
        ro = _entry_points(o, w, fb, fe, oracle_loader)
    except oracle_loader.OracleError as e:
        with pytest.raises(rsb.RsSyncError) as eg:
            _entry_points(g, w, fb, fe)
        assert (eg.value.code, eg.value.message) == (e.code, e.message)
        return
    _assert_same(_entry_points(g, w, fb, fe), ro)
