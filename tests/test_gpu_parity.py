"""Parity of the CUDA engine (through the C ABI) against the CPU oracle on identical seeded inputs.

Tolerances (north_star: argmin identical, loss-curve values and Sync delays within 1e-9 relative
in fp64).  Because engine and oracle implement the same arithmetic contract (DESIGN.md §3) the
observed differences are 0 or 1 ulp; the asserts use the stated 1e-9 bound for end results and a
tighter 1e-12 for single-stage probes.
"""
import numpy as np
import pytest

from conftest import rel_err, workload

pytestmark = pytest.mark.gpu

TOL = 1e-9        # north_star tolerance for loss-curve values and Sync delays
TOL_STAGE = 1e-12  # single-stage probes


@pytest.fixture(scope="module")
def pair_small(rsb, oracle_loader, w_small):
    g = rsb.SyncProblem(seed=100).load(w_small)
    o = oracle_loader.OracleProblem(threads=8, seed=100).load(w_small)
    return g, o, w_small


def test_log1p_bit_exact(rsb, oracle_loader):
    rng = np.random.default_rng(5)
    x = np.concatenate([
        10.0 ** rng.uniform(-320, 300, 20000), rng.uniform(0, 3, 20000), rng.uniform(0.35, 0.45, 5000),
        np.array([0.0, 1e-300, 2.0 ** -29, 2.0 ** -54, 0.41421356237309503, 1.0, 3.0, 2.0 ** 53, 1e308, np.inf]),
        2.0 ** rng.integers(-40, 60, 200).astype(np.float64) - 1.0 + 1.0])
    x = np.abs(x)
    a = rsb.probe_log1p(x)
    b = oracle_loader.log1p(x)
    assert np.array_equal(a, b)


def test_spline_records_bit_exact(pair_small):
    g, o, w = pair_small
    sr, q0, rec = g.probe_gyro()
    assert sr == w.gyro_rate and q0 == w.gyro_t0
    assert np.array_equal(rec, o.spline())


def test_problem_matrix_bit_exact(pair_small):
    g, o, w = pair_small
    n = w.n_rays
    for fid in (int(w.frame_ids[0]), int(w.frame_ids[17]), int(w.frame_ids[-1])):
        for delay in (-0.1, 0.0, 0.037, 0.0999):
            Pg = g.probe_problem_matrix(fid, delay, n)
            Po = o.problem_matrix(fid, delay, n)
            assert np.array_equal(Pg, Po), (fid, delay, rel_err(Pg, Po))


def test_problem_matrix_outside_gyro_span(pair_small):
    """timestamps + delay left of the first gyro sample, on the last spline segment, and beyond the
    end (the reference's right-side extrapolation quirk, minispline.cpp:48-55)"""
    g, o, w = pair_small
    n = w.n_rays
    nq = w.quats.shape[0]
    fid = int(w.frame_ids[5])
    t = float(w.ts_a[5].mean())
    t_end = w.gyro_t0 + (nq - 1) / w.gyro_rate
    for delay in (-1e3, w.gyro_t0 - t - 0.0004, w.gyro_t0 - t + 0.005, t_end - t - 0.02, t_end - t - 0.0101,
                  t_end - t + 0.0004, t_end - t + 0.0013, 1e3, 1e12):
        Pg = g.probe_problem_matrix(fid, delay, n)
        Po = o.problem_matrix(fid, delay, n)
        assert np.array_equal(Pg, Po, equal_nan=True), (delay, rel_err(Pg, Po))


def test_guess_motion_identical(pair_small):
    g, o, w = pair_small
    for fid in (int(w.frame_ids[3]), int(w.frame_ids[40])):
        for iters, stream in ((20, 1), (200, 3)):
            for call, off in ((0, 0), (3, 17)):
                mg, kg = g.probe_guess_motion(fid, 0.03, iters, stream, call, off)
                mo, ko = o.guess_motion(fid, 0.03, iters, stream, call, off)
                assert np.array_equal(mg, mo)
                assert kg == ko


def test_fp32_tournament_equals_exact_estimator(pair_small):
    """the product path (fp32 tournament, exact estimator when undecided) returns the exact binary64
    estimator's hypothesis bit for bit, and certifies most tasks without it"""
    g, o, w = pair_small
    exact_used = 0
    total = 0
    for fid in [int(f) for f in w.frame_ids[::7]]:
        for off, delay in enumerate(np.linspace(-0.08, 0.08, 9)):
            for iters, stream in ((20, 1), (200, 3)):
                mf, kf, used = g.probe_guess_motion_ex(fid, float(delay), iters, stream, 1, off, 0)
                me, ke, _ = g.probe_guess_motion_ex(fid, float(delay), iters, stream, 1, off, 2)
                assert np.array_equal(mf, me) and kf == ke, (fid, delay, iters)
                if iters == 20:
                    exact_used += used
                    total += 1
                    mo, ko = o.guess_motion(fid, float(delay), 20, 1, 1, off)
                    assert np.array_equal(mf, mo) and kf == ko
    assert exact_used <= 0.25 * total, (exact_used, total)


def test_estimator_degenerate_scenes(rsb, oracle_loader, synth_mod):
    """noise-free scene at the true delay (residuals ~1e-16, far below fp32 resolution) and a frame
    of identical rays (all rows zero): the tournament must hand over to the exact estimator and the
    curve must still match the oracle"""
    w = synth_mod.make_workload("tiny", noise_px=0.0, outlier_frac=0.0, true_delay=0.02)
    g = rsb.SyncProblem(seed=3).load(w)
    o = oracle_loader.OracleProblem(threads=2, seed=3).load(w)
    same = np.tile(w.rays_a[0][:1], (w.n_rays, 1))
    for p in (g, o):
        p.SetTrackResult(10 ** 4, w.ts_a[0], w.ts_a[0], same, same, w.n_rays)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    delays = np.array([0.0, 0.01, 0.02, 0.03])
    cg, flg = g.presync_grid(fb, fe, delays, call_no=2, return_flags=True)
    co, _, flo = o.presync_grid(fb, fe, delays, call_no=2, frame_costs=True)
    assert rel_err(cg, co) <= TOL and flg == flo
    st = g.stats()
    assert st["last_grid_tasks"] == 4 * w.n_frames
    # rows of norm < 1e-12 but finite: the exact estimator, and pre_sync's flags are the oracle's
    cz, flz = g.presync_grid(10 ** 4, 10 ** 4 + 1, delays, return_flags=True)
    coz, _, floz = o.presync_grid(10 ** 4, 10 ** 4 + 1, delays, frame_costs=True)
    assert np.array_equal(cz, coz) and flz == floz
    assert g.stats()["last_grid_exact_tasks"] == 4


def test_loss_and_gradient(pair_small):
    g, o, w = pair_small
    fid = int(w.frame_ids[10])
    m, k = o.guess_motion(fid, 0.036, 200, 3, 0, 0)
    l3, l5, grad = g.probe_loss(fid, 0.036, m, k)
    assert rel_err(l3, o.loss3(fid, 0.036, m, k)) <= TOL_STAGE
    l5o, go = o.loss5(fid, 0.036, m, k)
    assert rel_err(l5, l5o) <= TOL_STAGE
    assert np.max(np.abs(grad - go)) <= TOL_STAGE * max(1.0, np.max(np.abs(go)))
    # scale invariance of the loss in m: grad . m == 0 (SURVEY §8c pin 4)
    assert abs(np.dot(grad, m)) <= 1e-8 * np.linalg.norm(grad)


def test_lbfgs_matches_oracle(pair_small):
    g, o, w = pair_small
    for fid in (int(w.frame_ids[5]), int(w.frame_ids[33])):
        m0, k = o.guess_motion(fid, 0.036, 200, 3, 0, 0)
        mg, fg, itg, evg = g.probe_lbfgs(fid, 0.036, m0, k)
        mo, fo, ito, evo = o.lbfgs(fid, 0.036, m0, k)
        assert (itg, evg) == (ito, evo)
        assert rel_err(fg, fo) <= TOL_STAGE
        assert np.max(np.abs(mg - mo)) <= TOL_STAGE


def test_presync_curve_and_argmin(pair_small, rsb):
    g, o, w = pair_small
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[0]) + 60
    delays = rsb.presync_delays(0.0, w.presync_step, w.presync_radius)
    cg, flags = g.presync_grid(fb, fe, delays, call_no=7, return_flags=True)
    co = o.presync_grid(fb, fe, delays, call_no=7)
    assert flags == 0
    assert rel_err(cg, co) <= TOL
    assert int(np.argmin(cg)) == int(np.argmin(co))
    # known delay: argmin within one grid step of the truth (SURVEY §8c pin 7)
    assert abs(delays[int(np.argmin(cg))] - w.true_delay[0]) <= 1.5 * w.presync_step


def test_presync_api_matches_oracle(pair_small):
    g, o, w = pair_small
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    g.set_rng(100, 0)
    o.set_rng(100, 0)
    rg = g.PreSync(0.0, fb, fe, w.presync_step, w.presync_radius)
    ro = o.PreSync(0.0, fb, fe, w.presync_step, w.presync_radius)
    assert rg[1] == ro[1]                      # identical argmin delay (bit pattern of the grid point)
    assert rel_err(rg[0], ro[0]) <= TOL
    dg, cg = g.DebugPreSync(0.0, fb, fb + 30, 0.1, 51)
    do, co = o.DebugPreSync(0.0, fb, fb + 30, 0.1, 51)
    assert np.array_equal(dg, do)
    assert rel_err(cg, co) <= TOL
    assert g.call_counter() == 2


def test_presync_shard_equals_whole(pair_small, rsb):
    """offset-sharded evaluation (multi-GPU decomposition) reproduces the single call bit for bit."""
    g, o, w = pair_small
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[0]) + 20
    delays = rsb.presync_delays(0.0, 0.004, 0.1)
    whole = g.presync_grid(fb, fe, delays, call_no=3)
    parts = []
    for r in range(4):
        lo = len(delays) * r // 4
        hi = len(delays) * (r + 1) // 4
        parts.append(g.presync_grid(fb, fe, delays[lo:hi], call_no=3, offset_index_base=lo))
    assert np.array_equal(whole, np.concatenate(parts))


def test_sync_matches_oracle(pair_small):
    g, o, w = pair_small
    fb = int(w.frame_ids[0])
    fe = fb + 40
    g.set_rng(100, 10)
    o.set_rng(100, 10)
    dg = do = 0.038
    for i in range(2):
        cg, dg = g.Sync(dg, fb, fe, 0.0, 0.2)
        co, do, td, ts, cnt = o.Sync(do, fb, fe, 0.0, 0.2, trace=True)
        tdg, tsg = g.last_sync_trace()
        assert len(tdg) == len(td)
        assert rel_err(tdg, td) <= TOL
        assert rel_err(dg, do) <= TOL, (i, dg, do)
        assert rel_err(cg, co) <= TOL
        assert g.stats()["sync_lbfgs_evals"] == cnt[2]
    assert abs(dg - w.true_delay[0]) < 2e-3


def test_sync_batch_equals_sequence(pair_small):
    g, o, w = pair_small
    f0 = int(w.frame_ids[0])
    fbs = np.array([f0, f0 + 10, f0 + 20])
    fes = fbs + 30
    ini = np.array([0.036, 0.038, 0.040])
    g.set_rng(100, 50)
    seq = [g.Sync(float(ini[i]), int(fbs[i]), int(fes[i]), 0.0, 0.2) for i in range(3)]
    g.set_rng(100, 50)
    cb, db = g.sync_batch(ini, fbs, fes, 0.0, 0.2)
    assert np.array_equal(db, np.array([s[1] for s in seq]))
    assert np.array_equal(cb, np.array([s[0] for s in seq]))


def test_sync_batch_both_lbfgs_kernel_builds_and_any_lane_count(pair_small, monkeypatch):
    """the engine picks the L-BFGS kernel build (large / small blocks) by batch size and cuts the
    batch into lanes: neither may change a bit of any syncpoint's result"""
    g, o, w = pair_small
    f0 = int(w.frame_ids[0])
    fbs = np.array([f0 + 3 * i for i in range(9)])
    fes = fbs + 25
    ini = np.linspace(0.034, 0.040, 9)
    g.set_rng(100, 70)
    want = g.sync_batch(ini, fbs, fes, 0.0, 0.2)
    for build in ("small", "large"):
        monkeypatch.setenv("RSSYNC_LBFGS_BLOCKS", build)
        g.set_rng(100, 70)
        got = g.sync_batch(ini, fbs, fes, 0.0, 0.2)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    monkeypatch.delenv("RSSYNC_LBFGS_BLOCKS")
    co, do = o.sync_batch(ini, fbs, fes, 0.0, 0.2, call_nos=70 + np.arange(9, dtype=np.uint64))
    assert rel_err(want[1], do) <= TOL and rel_err(want[0], co) <= TOL


def test_ragged_and_sparse_frames(rsb, oracle_loader):
    """frames with different ray counts, gaps in the frame numbering, re-set frames"""
    w = workload("tiny")
    g = rsb.SyncProblem(seed=7)
    o = oracle_loader.OracleProblem(threads=2, seed=7)
    for p in (g, o):
        p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
    counts = [40, 33, 2, 17, 32, 40, 5, 31, 40, 9, 40, 40]
    for i, fid in enumerate(w.frame_ids):
        if i == 4:
            continue  # a skipped frame (README.md:66 of the reference)
        n = counts[i]
        for p in (g, o):
            p.SetTrackResult(int(fid), w.ts_a[i, :n], w.ts_b[i, :n], w.rays_a[i, :n], w.rays_b[i, :n], n)
    # replace one frame with a different ray count
    for p in (g, o):
        p.SetTrackResult(int(w.frame_ids[1]), w.ts_a[1, :40], w.ts_b[1, :40], w.rays_a[1, :40], w.rays_b[1, :40], 40)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    delays = np.linspace(-0.05, 0.05, 21)
    cg = g.presync_grid(fb, fe, delays)
    co = o.presync_grid(fb, fe, delays)
    assert rel_err(cg, co) <= TOL
    # empty range: the reference sums over no frames
    assert np.array_equal(g.presync_grid(10 ** 6, 10 ** 6 + 5, delays), np.zeros(21))
    g.set_rng(7, 3)
    o.set_rng(7, 3)
    rg = g.Sync(0.03, fb, fe, 0.0, 0.2)
    ro = o.Sync(0.03, fb, fe, 0.0, 0.2)
    assert rel_err(rg[1], ro[1]) <= TOL and rel_err(rg[0], ro[0]) <= TOL


@pytest.mark.parametrize("rays", [33, 64, 130, 224, 300, 500, 512])
def test_presync_ray_counts(rsb, oracle_loader, synth_mod, rays):
    """every SLOTS instantiation of the grid kernel (2..16 slots of 32 rays), ragged last slot"""
    w = synth_mod.make_workload("tiny", frames=6, rays=rays)
    g = rsb.SyncProblem(seed=11).load(w, bulk=True)
    o = oracle_loader.OracleProblem(threads=4, seed=11).load(w)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    delays = np.linspace(-0.03, 0.05, 23)
    cg = g.presync_grid(fb, fe, delays, call_no=4)
    co = o.presync_grid(fb, fe, delays, call_no=4)
    assert rel_err(cg, co) <= TOL
    assert int(np.argmin(cg)) == int(np.argmin(co))


def test_bulk_ingest_into_a_fresh_arena_that_grows(rsb, synth_mod):
    """a first bulk load larger than the arena's initial capacity (65 536 rays): the device arena
    grows while the batch's chunks are being ingested and must keep the chunks already there"""
    w = synth_mod.make_workload("tiny", frames=700, rays=200)
    a = rsb.SyncProblem(seed=3).load(w, bulk=True)
    b = rsb.SyncProblem(seed=3).load(w)  # frame by frame: host sort / transpose, one upload
    delays = np.linspace(-0.02, 0.02, 9)
    for lo in (0, 120, 350, 690):
        fb = int(w.frame_ids[lo])
        ca, fa = a.presync_grid(fb, fb + 8, delays, call_no=2, return_flags=True)
        cb, fl = b.presync_grid(fb, fb + 8, delays, call_no=2, return_flags=True)
        assert fa == 0 and fl == 0
        assert np.array_equal(ca, cb)


def test_bulk_ingest_ordering_against_single_frame_updates(rsb, synth_mod):
    """the bulk ingest runs on its own stream and the grid starts on the chunks that have landed:
    a frame set again after (before) the bulk call must win (lose), and grids over part of the
    frames must not disturb the rest"""
    w = synth_mod.make_workload("tiny", frames=130, rays=100)
    n = w.n_rays
    counts = np.full(w.n_frames, n)
    delays = np.linspace(-0.02, 0.02, 7)
    ids = [int(v) for v in w.frame_ids]
    k = 70  # the frame that is set twice, with frame 3's rays the second time
    # reference: frame by frame, final contents
    ref = rsb.SyncProblem(seed=9).load(w)
    ref.SetTrackResult(ids[k], w.ts_a[k], w.ts_b[k], w.rays_a[3], w.rays_b[3], n)
    want = ref.presync_grid(ids[0], ids[-1] + 1, delays, call_no=5)
    # bulk, then the single update
    a = rsb.SyncProblem(seed=9)
    a.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
    a.set_track_batch(w.frame_ids, counts, w.ts_a, w.ts_b, w.rays_a, w.rays_b)
    a.SetTrackResult(ids[k], w.ts_a[k], w.ts_b[k], w.rays_a[3], w.rays_b[3], n)
    assert np.array_equal(a.presync_grid(ids[0], ids[-1] + 1, delays, call_no=5), want)
    # the single (stale) version first, then the bulk with the final contents
    ra, rb = w.rays_a.copy(), w.rays_b.copy()
    ra[k], rb[k] = w.rays_a[3], w.rays_b[3]
    b = rsb.SyncProblem(seed=9)
    b.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
    b.SetTrackResult(ids[k], w.ts_a[k], w.ts_b[k], w.rays_a[k], w.rays_b[k], n)
    b.set_track_batch(w.frame_ids, counts, w.ts_a, w.ts_b, ra, rb)
    # grids over parts of the range, the last chunks first
    hi = b.presync_grid(ids[100], ids[-1] + 1, delays, call_no=5)
    lo = b.presync_grid(ids[0], ids[100], delays, call_no=5)
    assert np.array_equal(hi, ref.presync_grid(ids[100], ids[-1] + 1, delays, call_no=5))
    assert np.array_equal(lo, ref.presync_grid(ids[0], ids[100], delays, call_no=5))
    assert np.array_equal(b.presync_grid(ids[0], ids[-1] + 1, delays, call_no=5), want)


def test_presync_wide_delay_steps_use_global_path(rsb, oracle_loader, w_tiny):
    """delays 50 ms apart: the chunk's spline window does not fit the staging buffer, so phase A
    reads global memory; a 10 s offset leaves the gyro span entirely (spline edges)"""
    w = w_tiny
    g = rsb.SyncProblem(seed=5).load(w)
    o = oracle_loader.OracleProblem(threads=2, seed=5).load(w)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    delays = np.concatenate([np.arange(-0.3, 0.31, 0.05), [-10.0, 10.0]])
    cg, flags = g.presync_grid(fb, fe, delays, call_no=1, return_flags=True)
    co = o.presync_grid(fb, fe, delays, call_no=1)
    assert flags == 0
    assert rel_err(cg, co) <= TOL


def test_orientation_search_matches_oracle(rsb, oracle_loader, synth_mod):
    """core_testcode.cpp:184-233: PreSync under gyro_orientation variants; the true one wins"""
    w = workload("tiny", first_frame=200)  # non-negative microsecond timestamps (SURVEY a3)
    ts = w.gyro_t0 + np.arange(w.quats.shape[0]) / w.gyro_rate
    orients = ["yXz", "XYZ", "ZXY", "xyz", "XZy", "Yxz"]
    g = rsb.SyncProblem(seed=9).load(w)
    o = oracle_loader.OracleProblem(threads=2, seed=9).load(w)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    g.set_rng(9, 3)
    o.set_rng(9, 3)
    cg, dg = g.orientation_search(ts, w.omega, orients, 0.0, fb, fe, 0.005, 0.05)
    co, do = oracle_loader.orientation_search(o, ts, w.omega, orients, 0.0, fb, fe, 0.005, 0.05)
    assert np.array_equal(dg, do)
    assert rel_err(cg, co) <= TOL
    assert int(np.argmin(cg)) == 1
    assert g.call_counter() == 3 + len(orients)
    with pytest.raises(rsb.RsSyncError):
        g.orientation_search(ts, w.omega, ["XYZ", "XQZ"], 0.0, fb, fe, 0.005, 0.05)
    # explicit call numbers (what a rank of the sharded search passes): a subset of the variants in
    # one call reproduces their results of the full search and leaves the counter alone
    before = g.call_counter()
    sub = [4, 1, 2]
    cs, ds = g.orientation_search(ts, w.omega, [orients[k] for k in sub], 0.0, fb, fe, 0.005, 0.05,
                                  call_nos=np.array([3 + k for k in sub], dtype=np.uint64))
    assert np.array_equal(cs, cg[sub]) and np.array_equal(ds, dg[sub])
    assert g.call_counter() == before


def test_presync_windows_equals_sequence(pair_small):
    """several PreSync windows in one grid launch == the same PreSync calls one by one"""
    g, o, w = pair_small
    f0 = int(w.frame_ids[0])
    fbs = np.array([f0, f0 + 10, f0 + 25, f0 + 10, 10 ** 6])  # overlapping, repeated and empty windows
    fes = fbs + np.array([20, 30, 12, 30, 5])
    g.set_rng(100, 40)
    seq = [g.PreSync(0.0, int(a), int(b), 0.004, 0.08) for a, b in zip(fbs, fes)]
    g.set_rng(100, 40)
    c, d = g.presync_windows(0.0, fbs, fes, 0.004, 0.08)
    assert np.array_equal(c, [s[0] for s in seq]) and np.array_equal(d, [s[1] for s in seq])
    assert g.call_counter() == 45
    c3, d3 = g.presync_windows(0.0, fbs[:2], fes[:2], 0.004, 0.08, call_nos=np.array([40, 41], dtype=np.uint64))
    assert np.array_equal(c3, c[:2]) and np.array_equal(d3, d[:2])
    assert g.call_counter() == 45
    o.set_rng(100, 40)
    so = [o.PreSync(0.0, int(a), int(b), 0.004, 0.08) for a, b in zip(fbs[:3], fes[:3])]
    assert np.array_equal(d[:3], [x[1] for x in so]) and rel_err(c[:3], [x[0] for x in so]) <= TOL


def test_syncpoint_driver_matches_oracle(rsb, oracle_loader, w_small, tmp_path):
    """core_testcode's syncpoint loop (PreSync + 4 x Sync per syncpoint): the engine's batched,
    lock-step execution against the oracle issuing the reference's sequential calls"""
    import importlib
    driver = importlib.import_module("rs-sync_b200.driver")
    w = w_small
    cfg = driver.default_config(w, csv_path=str(tmp_path / "gpu.csv"))
    cfg["params"].update(sync_window=20, syncpoint_distance=20)
    cfg["input"].update(simple_presync_radius=60.0, simple_presync_step=4.0)
    g = rsb.SyncProblem(seed=100).load(w, bulk=True)
    o = oracle_loader.OracleProblem(threads=8, seed=100).load(w)
    rg = driver.run(g, cfg, mode="batched", debug_csv=str(tmp_path / "dbg.csv"), presync_delays=rsb.presync_delays)
    ro = driver.run(o, cfg, mode="sequential", debug_csv=str(tmp_path / "dbg_o.csv"))
    assert len(rg["syncpoints"]) == 3
    assert rel_err(rg["delay_ms"], ro["delay_ms"]) <= TOL
    assert rel_err(rg["cost"], ro["cost"]) <= TOL
    assert g.call_counter() == o.call_counter() == 1 + 3 * 5
    g2 = rsb.SyncProblem(seed=100).load(w, bulk=True)
    rs_ = driver.run(g2, cfg, mode="sequential", debug_csv=str(tmp_path / "dbg2.csv"))
    assert np.array_equal(rs_["delay_ms"], rg["delay_ms"])


def test_variable_rate_ingest_matches_oracle(rsb, oracle_loader, w_tiny):
    w = w_tiny
    rng = np.random.default_rng(3)
    # microsecond timestamps must be non-negative for the reference's unsigned arithmetic (SURVEY a3)
    ts = w.gyro_timestamps_us() + 10_000_000 + rng.integers(-150, 150, w.quats.shape[0])
    ts = np.sort(ts)
    g = rsb.SyncProblem()
    o = oracle_loader.OracleProblem()
    g.SetGyroQuaternions(ts, w.quats, len(ts))
    o.SetGyroQuaternions(ts, w.quats, len(ts))
    sr, q0, rec = g.probe_gyro()
    qo, sro, q0o = o.resampled()
    assert sr == sro == 1000.0 and q0 == q0o
    assert np.array_equal(rec, o.spline())


def test_error_conventions(rsb, w_tiny):
    w = w_tiny
    g = rsb.SyncProblem()
    with pytest.raises(rsb.RsSyncError) as e:
        g.PreSync(0.0, 0, 10, 0.002, 0.1)
    assert e.value.code == rsb.E_STATE
    bad = w.rays_a[0].copy()
    bad[3, 1] = np.nan
    with pytest.raises(rsb.RsSyncError) as e:
        g.SetTrackResult(1, w.ts_a[0], w.ts_b[0], bad, w.rays_b[0], w.n_rays)
    assert e.value.code == rsb.E_NONFINITE and e.value.message == "set-track-result: non-finite numbers in rays_a"
    tsb = w.ts_b[0].copy()
    tsb[0] = np.inf
    with pytest.raises(rsb.RsSyncError) as e:
        g.SetTrackResult(1, w.ts_a[0], tsb, w.rays_a[0], w.rays_b[0], w.n_rays)
    assert e.value.message == "set-track-result: non-finite numbers in ts_b"
    ts = w.gyro_timestamps_us().copy()
    ts[5], ts[6] = ts[6], ts[5]
    with pytest.raises(rsb.RsSyncError) as e:
        g.SetGyroQuaternions(ts, w.quats, len(ts))
    assert e.value.code == rsb.E_ORDER
    assert e.value.message == f"set-gyro-quaternions:  timestamps out of order at pos 6 ({ts[5]} > {ts[6]})"
    # non-finite gyro -> non-finite P flagged by the kernel, PreSync reports the reference's message
    q = w.quats.copy()
    q[len(q) // 2] = np.nan
    g.SetGyroQuaternions(q, len(q), w.gyro_rate, w.gyro_t0)
    g.SetTrackResult(int(w.frame_ids[0]), w.ts_a[0], w.ts_b[0], w.rays_a[0], w.rays_b[0], w.n_rays)
    with pytest.raises(rsb.RsSyncError) as e:
        g.PreSync(0.0, int(w.frame_ids[0]), int(w.frame_ids[0]) + 1, 0.005, 0.05)
    assert e.value.code == rsb.E_NONFINITE and e.value.message == "pre-sync: non-finite numbers in P"


def test_golden_fixture(rsb, w_tiny):
    """CUDA path against the committed golden vectors (tests/golden/tiny_curve.json)"""
    import json, os
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "tiny_curve.json")))
    w = w_tiny
    p = rsb.SyncProblem(seed=100).load(w)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    delays = rsb.presync_delays(0.0, w.presync_step, w.presync_radius)
    assert [float(d).hex() for d in delays] == g["delays_hex"]
    costs = p.presync_grid(fb, fe, delays, call_no=0)
    want = np.array([float.fromhex(h) for h in g["costs_hex"]])
    assert rel_err(costs, want) <= TOL
    assert int(np.argmin(costs)) == int(np.argmin(want))
    p.set_rng(100, 1)
    sc, sd = p.Sync(0.035, fb, fe - 1, 0.0, 0.2)
    assert rel_err(sd, float.fromhex(g["sync_delay_hex"])) <= TOL
    assert rel_err(sc, float.fromhex(g["sync_cost_hex"])) <= TOL


def test_cxx_dropin_runs_like_the_c_abi(rsb, w_tiny, tmp_path):
    """a C++ caller written against the reference's ISyncProblem interface (include/rssync.h), run
    on the GPU through CreateSyncProblem's vtable, returns what the C ABI returns"""
    import os, struct, subprocess
    from conftest import ROOT
    w = w_tiny
    blob = tmp_path / "workload.bin"
    with open(blob, "wb") as f:
        f.write(struct.pack("<qqqdd", w.quats.shape[0], w.n_frames, w.n_rays, w.gyro_rate, w.gyro_t0))
        f.write(np.ascontiguousarray(w.quats).tobytes())
        f.write(np.ascontiguousarray(w.frame_ids).tobytes())
        for a in (w.ts_a, w.ts_b, w.rays_a, w.rays_b):
            f.write(np.ascontiguousarray(a).tobytes())
    src = tmp_path / "caller.cpp"
    src.write_text(r'''
#include <rssync.h>
#include <cstdio>
#include <cstdint>
#include <memory>
#include <vector>
int main(int, char** argv) {
    FILE* f = std::fopen(argv[1], "rb");
    int64_t nq, nf, nr; double rate, t0;
    if (!f || std::fread(&nq, 8, 1, f) != 1 || std::fread(&nf, 8, 1, f) != 1 || std::fread(&nr, 8, 1, f) != 1 ||
        std::fread(&rate, 8, 1, f) != 1 || std::fread(&t0, 8, 1, f) != 1) return 2;
    std::vector<double> q(4 * nq), tsa(nf * nr), tsb(nf * nr), ra(3 * nf * nr), rb(3 * nf * nr);
    std::vector<int64_t> ids(nf);
    if (std::fread(q.data(), 8, q.size(), f) != q.size() || std::fread(ids.data(), 8, nf, f) != (size_t)nf ||
        std::fread(tsa.data(), 8, tsa.size(), f) != tsa.size() || std::fread(tsb.data(), 8, tsb.size(), f) != tsb.size() ||
        std::fread(ra.data(), 8, ra.size(), f) != ra.size() || std::fread(rb.data(), 8, rb.size(), f) != rb.size()) return 3;
    std::unique_ptr<ISyncProblem> sp{CreateSyncProblem()};   // core_testcode.cpp:248
    sp->SetGyroQuaternions(q.data(), (size_t)nq, rate, t0);
    for (int64_t i = 0; i < nf; ++i)
        sp->SetTrackResult(ids[i], &tsa[i * nr], &tsb[i * nr], &ra[3 * i * nr], &rb[3 * i * nr], (size_t)nr);
    std::vector<double> dd(11), cc(11);
    sp->DebugPreSync(0.0, ids[0], ids[0] + nf, 0.05, dd.data(), cc.data(), 11);
    auto p = sp->PreSync(0.0, ids[0], ids[0] + nf, 0.005, 0.05);
    auto s = sp->Sync(p.second, ids[0], ids[0] + nf - 1, 0.0, 0.05);
    std::printf("%a %a %a %a %a %a\n", p.first, p.second, s.first, s.second, dd[3], cc[3]);
    return 0;
}
''')
    exe = tmp_path / "caller"
    libdir = os.path.dirname(rsb.LIB_PATH)
    r = subprocess.run(["g++", "-std=c++17", f"-I{ROOT}/include", str(src), "-o", str(exe), f"-L{libdir}",
                        "-lrssync_b200", f"-Wl,-rpath,{libdir}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe), str(blob)], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0, r.stderr
    got = [float.fromhex(x) for x in r.stdout.split()]
    g = rsb.SyncProblem(seed=100).load(w)
    fb, nf = int(w.frame_ids[0]), w.n_frames
    dd, cc = g.DebugPreSync(0.0, fb, fb + nf, 0.05, 11)
    p = g.PreSync(0.0, fb, fb + nf, 0.005, 0.05)
    s = g.Sync(p[1], fb, fb + nf - 1, 0.0, 0.05)
    assert got == [p[0], p[1], s[0], s[1], dd[3], cc[3]]


def test_pixel_front_end_matches_host_rays(rsb, oracle_loader, synth_mod):
    """rssync_set_track_pixels (undistort + rolling-shutter timestamps + unit rays + sort on the device,
    core_testcode.cpp:63-95,134-161) against the same frames fed as host-computed rays: identical
    timestamps / ordering, rays equal up to the rounding of tan / cos"""
    w = synth_mod.make_workload("tiny", rays=130)
    counts = np.full(w.n_frames, w.n_rays)
    ta, tb = w.frame_ids / w.fps, (w.frame_ids + 1) / w.fps
    assert np.array_equal(w.ts_a, ta[:, None] + synth_mod.READOUT * (w.px_a[..., 1] / synth_mod.HEIGHT))
    ref = rsb.SyncProblem(seed=21).load(w, bulk=True)
    pix = rsb.SyncProblem(seed=21)
    pix.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
    half = w.n_frames // 2  # two calls: the second grows the device arena, contents preserved
    for sl in (slice(0, half), slice(half, None)):
        pix.set_track_pixels(w.frame_ids[sl], counts[sl], ta[sl], tb[sl], w.px_a[sl], w.px_b[sl], synth_mod.LENS,
                             synth_mod.HEIGHT)
    assert pix.stats()["frames"] == w.n_frames and pix.stats()["rays"] == w.n_frames * w.n_rays
    for fid in (int(w.frame_ids[0]), int(w.frame_ids[-1])):
        a = ref.probe_problem_matrix(fid, 0.02, w.n_rays)
        b = pix.probe_problem_matrix(fid, 0.02, w.n_rays)
        assert np.max(np.abs(a - b)) <= 1e-13 * np.max(np.abs(a))
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    delays = np.linspace(-0.04, 0.06, 26)
    ca = ref.presync_grid(fb, fe, delays, call_no=2)
    cb = pix.presync_grid(fb, fe, delays, call_no=2)
    assert rel_err(cb, ca) <= TOL and int(np.argmin(ca)) == int(np.argmin(cb))
    # a host-side ray frame may replace / follow device-ingested ones
    pix.SetTrackResult(int(w.frame_ids[1]), w.ts_a[1], w.ts_b[1], w.rays_a[1], w.rays_b[1], w.n_rays)
    assert rel_err(pix.presync_grid(fb, fe, delays, call_no=2), ca) <= TOL
    o = oracle_loader.OracleProblem(threads=2, seed=21).load(w)
    assert rel_err(cb, o.presync_grid(fb, fe, delays, call_no=2)) <= TOL
    with pytest.raises(rsb.RsSyncError):
        pix.set_track_pixels(w.frame_ids[:1], counts[:1], ta[:1], tb[:1], w.px_a[:1], w.px_b[:1],
                             (0.01, 0.0, 1.0, 0, 0, 0, 0, 0, 0), synth_mod.HEIGHT)


def test_adopted_device_state_reproduces_the_source(rsb, w_small):
    """replication without re-ingesting (what bench.py does across ranks with an NCCL broadcast and
    rssync_create_multi does inside the library): a second problem adopts the frame table and sizes,
    its buffers are filled device-to-device, and every result equals the source's bit for bit"""
    import importlib
    import torch
    sharded = importlib.import_module("rs-sync_b200.sharded")
    w = w_small
    a = rsb.SyncProblem(seed=100).load(w, bulk=True)
    ft = a.frame_table()
    assert ft.shape[0] == w.n_frames and np.array_equal(ft["id"], w.frame_ids) and np.all(ft["n"] == w.n_rays)
    src, st = sharded.device_buffers(a)
    b = rsb.SyncProblem(seed=100)
    b.adopt_state(ft, st["arena_rays"], st["gyro_samples"], st["sample_rate"], st["first_timestamp"])
    dst, st_b = sharded.device_buffers(b)
    for k in src:
        assert dst[k].data_ptr() != src[k].data_ptr() and dst[k].numel() == src[k].numel()
        dst[k].copy_(src[k])
    torch.cuda.synchronize()
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    delays = np.linspace(-0.05, 0.05, 21)
    assert np.array_equal(a.presync_grid(fb, fe, delays, call_no=2), b.presync_grid(fb, fe, delays, call_no=2))
    for p in (a, b):
        p.set_rng(100, 30)
    assert a.Sync(0.038, fb, fb + 30, 0.0, 0.2) == b.Sync(0.038, fb, fb + 30, 0.0, 0.2)
    # the adopting problem stays a full problem: a frame set afterwards lands in its own arena
    for p in (a, b):
        p.SetTrackResult(10 ** 5, w.ts_a[3], w.ts_b[3], w.rays_a[3], w.rays_b[3], w.n_rays)
    assert np.array_equal(a.presync_grid(10 ** 5, 10 ** 5 + 1, delays), b.presync_grid(10 ** 5, 10 ** 5 + 1, delays))
    assert b.stats()["frames"] == w.n_frames + 1


def test_pipelined_replication_behind_a_bulk_ingest(rsb, w_small, synth_mod):
    """the pipelined form (sharded.replicate_state across ranks): the source has just taken a bulk
    SetTrackResult whose chunks are still in flight; each chunk is copied on, on a side stream, as soon
    as it has landed, and the adopting problem's grid starts behind the chunks it was told to expect"""
    import importlib
    import torch
    sharded = importlib.import_module("rs-sync_b200.sharded")
    w = w_small
    counts = np.full(w.n_frames, w.n_rays)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    delays = np.linspace(-0.05, 0.05, 21)
    a = rsb.SyncProblem(seed=100).load(w, bulk=True)
    want = a.presync_grid(fb, fe, delays, call_no=2)
    b = rsb.SyncProblem(seed=100)
    side = torch.cuda.Stream()
    w2 = synth_mod.make_workload("small", seed=9)
    fresh = rsb.SyncProblem(seed=100)  # its first ingest, into an arena that grows on the way
    for rep, (a, ww) in enumerate(((a, w), (a, w2), (a, w), (fresh, w))):
        a.SetGyroQuaternions(ww.quats, ww.quats.shape[0], ww.gyro_rate, ww.gyro_t0)
        a.set_track_batch(ww.frame_ids, counts, ww.ts_a, ww.ts_b, ww.rays_a, ww.rays_b)
        st = a.device_state_pipelined()
        chunks = st["chunks"]
        assert chunks and all(lo < hi <= st["arena_rays"] for lo, hi in chunks)
        b.adopt_state(a.frame_table(), st["arena_rays"], st["gyro_samples"], st["sample_rate"], st["first_timestamp"])
        dst, _ = sharded.device_buffers(b)
        src = {k: torch.as_tensor(sharded._DevicePtr(*st[k]), device="cuda") for k in ("rays", "orig", "pos", "spline_records")}
        skip = 3 if rep == 2 else 0
        if skip:  # as if the first chunks were no longer in flight (an ingest that had to wait for them)
            torch.cuda.synchronize()
        pieces = [(k if k < 0 else k + skip, lo, hi)
                  for k, lo, hi in sharded._merge_chunks(chunks[skip:], 3, st["arena_rays"])]
        assert pieces[-1][0] == len(chunks) - 1 and (pieces[0][0] == -1) == bool(skip)
        covered = np.zeros(st["arena_rays"], dtype=bool)  # every ray of the arena is in some piece
        for _, lo, hi in pieces:
            covered[lo:hi] = True
        assert covered.all()
        with torch.cuda.stream(side):
            a.stream_wait_chunk(-1, side.cuda_stream)
            dst["spline_records"].copy_(src["spline_records"], non_blocking=True)
            b.expect_chunk(0, st["arena_rays"], side.cuda_stream)
            for k_last, lo, hi in pieces:
                if k_last >= 0:
                    a.stream_wait_chunk(k_last, side.cuda_stream)
                for name, width in (("rays", 64), ("orig", 4), ("pos", 4)):
                    dst[name][lo * width:hi * width].copy_(src[name][lo * width:hi * width], non_blocking=True)
                b.expect_chunk(lo, hi, side.cuda_stream)
            a.note_reader(side.cuda_stream)
        ga = a.presync_grid(fb, fe, delays, call_no=2)
        gb = b.presync_grid(fb, fe, delays, call_no=2)
        assert np.array_equal(ga, gb)
        assert np.array_equal(ga, want) == (rep != 1)
    with pytest.raises(rsb.RsSyncError):
        a.stream_wait_chunk(99, side.cuda_stream)


def test_simplified_loss_mode_matches_oracle(rsb, oracle_loader, w_small):
    """the thesis' simplified (no-translation) loss mode (rssync_set_loss_mode): PreSync curve, argmin
    and the whole Sync trajectory equal the oracle's; switching back restores the reference's loss"""
    w = w_small
    g = rsb.SyncProblem(seed=100).load(w, bulk=True)
    o = oracle_loader.OracleProblem(threads=8, seed=100).load(w)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    full = g.DebugPreSync(0.0, fb, fe, 0.1, 41)[1]
    for p in (g, o):
        p.set_loss_mode(True)
        p.set_rng(100, 7)
    dg, cg = g.DebugPreSync(0.0, fb, fe, 0.1, 41)
    do, co = o.DebugPreSync(0.0, fb, fe, 0.1, 41)
    assert np.array_equal(dg, do) and rel_err(cg, co) <= TOL
    assert int(np.argmin(cg)) == int(np.argmin(co))
    assert abs(dg[int(np.argmin(cg))] - w.true_delay[0]) <= 0.005
    assert not np.allclose(cg, full)
    pg = g.PreSync(0.0, fb, fe, w.presync_step, w.presync_radius)
    po = o.PreSync(0.0, fb, fe, w.presync_step, w.presync_radius)
    assert pg[1] == po[1] and rel_err(pg[0], po[0]) <= TOL
    sg = g.Sync(pg[1], fb, fb + 40, 0.0, 0.2)
    so = o.Sync(po[1], fb, fb + 40, 0.0, 0.2, trace=True)
    tdg, _ = g.last_sync_trace()
    assert len(tdg) == len(so[2]) and rel_err(tdg, so[2]) <= TOL
    assert rel_err(sg[1], so[1]) <= TOL and rel_err(sg[0], so[0]) <= TOL
    assert abs(sg[1] - w.true_delay[0]) < 3e-3
    st = g.stats()
    assert st["sync_lbfgs_evals"] == 0 and st["sync_init_tasks"] == 0 and st["sync_row_builds"] > 0
    # a batch, windows in one launch
    fbs = np.array([fb, fb + 12])
    cb, db = g.sync_batch(np.array([0.036, 0.039]), fbs, fbs + 30, 0.0, 0.2)
    cbo, dbo = o.sync_batch(np.array([0.036, 0.039]), fbs, fbs + 30, 0.0, 0.2)
    assert rel_err(db, dbo) <= TOL and rel_err(cb, cbo) <= TOL
    g.set_loss_mode(False)
    assert np.array_equal(g.DebugPreSync(0.0, fb, fe, 0.1, 41)[1] != cg, np.ones(41, dtype=bool))


def test_device_gyro_ingest_matches_host_and_oracle(rsb, oracle_loader, synth_mod):
    """the gyro ingest on the device (engine.cu K8): the contract's trig functions, the blocked
    integration scan, the variable-rate resampling and the spline elimination sweeps give the bits of
    the engine's host code and of the oracle"""
    rng = np.random.default_rng(4)
    xs = np.concatenate([rng.uniform(-3.3, 3.3, 50000), rng.uniform(0, 0.2, 20000), rng.uniform(-50, 50, 20000)])
    for which in ("sin", "cos"):
        assert np.array_equal(rsb.probe_spec_trig(xs, which, on_device=True), rsb.probe_spec_trig(xs, which))
    ys = np.concatenate([rng.uniform(-1, 1, 50000), 1 - rng.uniform(0, 1e-6, 20000) ** 2, [1.0, -1.0, 0.5, 1.0000000000000002]])
    assert np.array_equal(rsb.probe_spec_trig(ys, "acos", on_device=True), rsb.probe_spec_trig(ys, "acos"), equal_nan=True)
    # variable-rate SetGyroQuaternions: a 450 Hz track with jitter, an unaligned first timestamp, 3 blocks of
    # resampled samples; records == oracle's (resampled samples included)
    n = 1700
    ts = (7_000_123 + np.cumsum(rng.integers(2100, 2350, n))).astype(np.int64)
    q = rng.normal(size=(n, 4)) * 0.05 + np.array([1.0, 0, 0, 0])
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    q[::7] *= -1  # sign flips: slerp takes the short way (quat.cpp:58-60)
    g = rsb.SyncProblem()
    o = oracle_loader.OracleProblem()
    g.SetGyroQuaternions(ts, q, n)
    o.SetGyroQuaternions(ts, q, n)
    sr, q0, rec = g.probe_gyro()
    qo, sro, q0o = o.resampled()
    assert sr == sro == 450.0 and q0 == q0o
    assert np.array_equal(rec[:, 0:4], qo)
    assert np.array_equal(rec, o.spline())
    # a non-finite sample after interpolation is the reference's panic (core_private.cpp:180-181)
    # (a dot product above 1 is NOT one: acos gives NaN, `theta > 1e-9` is false and quat_slerp falls
    # back to the linear weights, quat.cpp:61-70 -- same here)
    odd = q.copy()
    odd[900] = [2.0, 0, 0, 0]
    g.SetGyroQuaternions(ts, odd, n)
    o.SetGyroQuaternions(ts, odd, n)
    assert np.array_equal(g.probe_gyro()[2], o.spline())
    g.SetGyroQuaternions(ts, q, n)
    bad = q.copy()
    bad[900, 2] = np.inf
    with pytest.raises(rsb.RsSyncError) as e:
        g.SetGyroQuaternions(ts, bad, n)
    assert e.value.code == rsb.E_NONFINITE and "non-finite sample after interpolation" in e.value.message
    with pytest.raises(oracle_loader.OracleError):
        o.SetGyroQuaternions(ts, bad, n)
    # the problem still holds the good track
    assert np.array_equal(g.probe_gyro()[2], rec)


def test_orientation_search_long_track_all_variants(rsb, oracle_loader, synth_mod):
    """all 48 variants on a track of several scan blocks, through the device pipeline (integration,
    resampling, elimination, records, grids queued back to back), against the oracle's loop of host
    calls; the search leaves the problem holding the last variant's gyro"""
    w = workload("small")
    ts = w.gyro_t0 + np.arange(w.quats.shape[0]) / w.gyro_rate
    assert w.quats.shape[0] > 3 * 512
    orients = synth_mod.ORIENTATIONS
    g = rsb.SyncProblem(seed=100).load(w, bulk=True)
    o = oracle_loader.OracleProblem(threads=8, seed=100).load(w)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[0]) + 24
    g.set_rng(100, 5)
    o.set_rng(100, 5)
    cg, dg = g.orientation_search(ts, w.omega, orients, 0.0, fb, fe, 0.004, 0.06)
    co, do = oracle_loader.orientation_search(o, ts, w.omega, orients, 0.0, fb, fe, 0.004, 0.06)
    assert np.array_equal(dg, do) and rel_err(cg, co) <= TOL
    assert orients[int(np.argmin(cg))] == "XYZ"
    assert g.call_counter() == o.call_counter() == 5 + 48
    assert np.array_equal(g.probe_gyro()[2], o.spline())
    # the integration on the device equals the host function of the C ABI
    qh = rsb.integrate_gyro(ts, w.omega, orients[-1])
    g2 = rsb.SyncProblem()
    g2.SetGyroQuaternions((ts * 1000000).astype(np.int64), qh, len(ts))
    assert np.array_equal(g2.probe_gyro()[2], g.probe_gyro()[2])
