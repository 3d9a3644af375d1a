"""Every kernel instantiation and ragged frame layout of the engine against the CPU oracle (bit for
bit, or the north_star's 1e-9 for Sync) and against the independent long-double reference of
tests/plain_reference.py (under its per-value bound).

The estimator kernels are instantiated at SLOTS in {2, 4, 6, 7, 8, 12, 16} (slots_for in
engine.cu) by the widest frame a call selects.  The ray counts below sit on both sides of every
boundary and at the quartile-rank edges; single-frame grids give one (delay, frame) cell per value.
Then: one bulk batch whose frames range from 2 to 512 rays (the widest instantiation serving narrow
frames), rays whose ts_a tie (the sort's tie-break fixes the summation order), delays that put
rays at the edges of the gyro span, and degenerate frames.  The largest bound ratio per stage is
printed at the end (run with -s).
"""
import numpy as np
import pytest

import plain_reference as ref
from conftest import rel_err, workload

pytestmark = pytest.mark.gpu

TOL = 1e-9
SEED = 29
RAY_COUNTS = [2, 3, 4, 5, 31, 32, 33, 64, 65, 128, 129, 192, 193, 224, 225, 256, 257, 384, 385, 512]
# one or two counts per SLOTS value of the Sync kernels (2 4 6 7 8 12 16), both quartile-rank edges
SYNC_COUNTS = [3, 33, 65, 128, 129, 193, 225, 256, 257, 385, 512]
GRID_WARPS = 8  # RS_GRID_WARPS: a unit of fewer delays than this runs unstaged
LOG = ref.RatioLog()


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("\nplain reference vs engine, largest bound ratio per stage:", LOG.report())


_PAIRS = {}


def pair(rsb, oracle_loader, n, frames=2):
    key = (n, frames)
    if key not in _PAIRS:
        w = workload("tiny", frames=frames, rays=n, seed=SEED)
        g = rsb.SyncProblem(seed=SEED).load(w)
        o = oracle_loader.OracleProblem(threads=8, seed=SEED).load(w)
        _PAIRS[key] = (g, o, w, g.probe_gyro()[2])
    return _PAIRS[key]


def mode(ps, simplified):
    for p in ps:
        p.set_loss_mode(simplified)


# ------------------------------------------------------------------------------------------------
# C.1  ray-count matrix


@pytest.mark.parametrize("n", RAY_COUNTS)
def test_probes_against_plain_reference(rsb, oracle_loader, n):
    """problem matrix, estimator (product path and exact binary64, 20 and 200 hypotheses), k,
    Loss3 / Loss5 / gradient and L-BFGS at every ray count"""
    g, o, w, rec = pair(rsb, oracle_loader, n)
    mode((g, o), False)
    assert np.array_equal(rec, o.spline())
    for i in range(w.n_frames):
        fid = int(w.frame_ids[i])
        for off, delay in enumerate((0.0, 0.037)):
            P = ref.frame_rows(rec, w.gyro_t0, w.gyro_rate, delay, w, i)
            Pg = g.probe_problem_matrix(fid, delay, n)
            assert np.array_equal(Pg, o.problem_matrix(fid, delay, n))
            assert LOG.add("rows", ref.ratio(Pg, P.astype(np.float64), ref.E)) <= 1.0
            for iters, stream in ((20, 1), (200, 3)):
                est = ref.Estimate(P, ref.rng_task_key(SEED, stream, 4, off, fid), iters)
                mo, ko = o.guess_motion(fid, delay, iters, stream, 4, off)
                for m_ in (0, 2):
                    mg, kg, _ = g.probe_guess_motion_ex(fid, delay, iters, stream, 4, off, m_)
                    assert np.array_equal(mg, mo) and kg == ko, (fid, delay, iters, m_)
                d = [ref.ratio(mg, est.hyp[t].astype(np.float64), est.dM[t]) for t in est.near]
                assert LOG.add("estimator", min(d)) <= 1.0, (fid, delay, iters, est.near)
                t = est.near[int(np.argmin(d))]
                _, _, kr, dk = ref.presync_cost(P, est.hyp[t], float(est.dM[t]))
                assert LOG.add("k", ref.ratio(kg, kr, dk)) <= 1.0
                l3, l5, gr = g.probe_loss(fid, delay, mg, kg)
                r3, b3 = ref.loss3(P, mg, kg)
                r5, rg, b5, bg = ref.loss5(P, mg, kg)
                assert LOG.add("loss3", ref.ratio(l3, r3, b3)) <= 1.0
                assert LOG.add("loss5", ref.ratio(l5, r5, b5)) <= 1.0
                assert LOG.add("gradient", ref.ratio(gr, rg, bg)) <= 1.0
                if iters == 200:
                    # L-BFGS (the restated ensmallen, unpinned): the oracle's result, and a descent
                    # of the reference's objective
                    m1, f1, it, ev = g.probe_lbfgs(fid, delay, mg, kg)
                    mo1, fo1, ito, evo = o.lbfgs(fid, delay, mo, ko)
                    assert (it, ev) == (ito, evo) and rel_err(f1, fo1) <= 1e-12
                    assert np.max(np.abs(m1 - mo1)) <= 1e-12
                    L1, g1, b1, _ = ref.loss5(P, m1, kg)
                    assert L1 <= r5 + b1 + b5
                    # f is the objective at the last trial of the last line search; where that was
                    # the accepted step it is the reference's value at m, and the gradient test
                    # stopped the iteration unless the cap did
                    if abs(f1 - L1) <= b1:
                        LOG.add("lbfgs", ref.ratio(f1, L1, b1))
                        assert np.linalg.norm(g1) <= 1e-4 or it == 200, (n, fid, delay, it, ev)


@pytest.mark.parametrize("simplified", [False, True], ids=["full", "simplified"])
@pytest.mark.parametrize("n", RAY_COUNTS)
def test_presync_cells_against_plain_reference(rsb, oracle_loader, n, simplified):
    """presync_kernel<SLOTS, SIMPLE> at every ray count, cell by cell: a single-frame grid gives the
    frame's cost per delay (its double-double sum over one frame is exact).  16 delays 1 ms apart
    run staged (units of >= GRID_WARPS delays), 5 delays unstaged."""
    g, o, w, rec = pair(rsb, oracle_loader, n)
    mode((g, o), simplified)
    stage = "presync_simplified" if simplified else "presync"
    for i in range(w.n_frames):
        fid = int(w.frame_ids[i])
        for delays in (0.03 + 0.001 * np.arange(2 * GRID_WARPS), np.array([-0.04, -0.01, 0.0, 0.02, 0.045])):
            cg, flags = g.presync_grid(fid, fid + 1, delays, call_no=6, offset_index_base=3, return_flags=True)
            co = o.presync_grid(fid, fid + 1, delays, call_no=6, offset_index_base=3)
            assert flags == 0
            assert np.array_equal(cg, co), (fid, rel_err(cg, co))
            for d, delay in enumerate(delays):
                P = ref.frame_rows(rec, w.gyro_t0, w.gyro_rate, delay, w, i)
                cands = ref.presync_cell(P, ref.rng_task_key(SEED, 1, 6, 3 + d, fid), simplified)
                assert LOG.add(stage, ref.cell_ratio(cg[d], cands)) <= 1.0, (fid, delay)
    mode((g, o), False)


@pytest.mark.parametrize("simplified", [False, True], ids=["full", "simplified"])
@pytest.mark.parametrize("n", SYNC_COUNTS)
def test_sync_at_every_instantiation(rsb, oracle_loader, monkeypatch, n, simplified):
    """sync_init_kernel<SLOTS> and sync_motion_fgrad_kernel<SLOTS, small / large blocks> against
    the oracle: Sync with its trace, and sync_batch under both L-BFGS kernel builds"""
    g, o, w, _ = pair(rsb, oracle_loader, n, frames=6)
    mode((g, o), simplified)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1])  # Sync's frame_end is inclusive
    for p in (g, o):
        p.set_rng(SEED, 5)
    cg, dg = g.Sync(0.035, fb, fe, 0.0, 0.2)
    tdg, _ = g.last_sync_trace()
    evals = g.stats()["sync_lbfgs_evals"]
    co, do, td, _, cnt = o.Sync(0.035, fb, fe, 0.0, 0.2, trace=True)
    assert len(tdg) == len(td) and rel_err(tdg, td) <= TOL
    assert rel_err(dg, do) <= TOL and rel_err(cg, co) <= TOL
    assert evals == cnt[2]
    for build in ("small", "large"):
        monkeypatch.setenv("RSSYNC_LBFGS_BLOCKS", build)
        cb, db = g.sync_batch(np.array([0.035]), [fb], [fe], 0.0, 0.2, call_nos=np.array([5], dtype=np.uint64))
        assert rel_err(db, [do]) <= TOL and rel_err(cb, [co]) <= TOL, build
    monkeypatch.delenv("RSSYNC_LBFGS_BLOCKS")
    mode((g, o), False)


# ------------------------------------------------------------------------------------------------
# C.2  mixed widths in one bulk batch

MIXED = [2, 3, 17, 33, 100, 225, 385, 512]


@pytest.fixture(scope="module")
def mixed(rsb, oracle_loader):
    """72 frames (the device-ingest path takes >= 64) of 2 to 512 rays, bulk and frame by frame"""
    w = workload("tiny", frames=72, rays=512, seed=SEED)
    counts = np.array([MIXED[(5 * i) % len(MIXED)] for i in range(w.n_frames)])
    cat = [np.concatenate([a[i, :counts[i]] for i in range(w.n_frames)]) for a in (w.ts_a, w.ts_b, w.rays_a, w.rays_b)]
    bulk = rsb.SyncProblem(seed=SEED)
    bulk.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
    bulk.set_track_batch(w.frame_ids, counts, *cat)
    fbf = rsb.SyncProblem(seed=SEED)
    o = oracle_loader.OracleProblem(threads=8, seed=SEED)
    for p in (fbf, o):
        p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
        for i, fid in enumerate(w.frame_ids):
            c = int(counts[i])
            p.SetTrackResult(int(fid), w.ts_a[i, :c], w.ts_b[i, :c], w.rays_a[i, :c], w.rays_b[i, :c], c)
    return bulk, fbf, o, w, counts


def test_mixed_widths_grid_windows_and_sync(mixed):
    bulk, fbf, o, w, counts = mixed
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    for delays in (0.03 + 0.001 * np.arange(2 * GRID_WARPS), np.array([-0.02, 0.01, 0.04])):
        cb = bulk.presync_grid(fb, fe, delays, call_no=2)
        assert np.array_equal(cb, fbf.presync_grid(fb, fe, delays, call_no=2))
        assert rel_err(cb, o.presync_grid(fb, fe, delays, call_no=2)) <= TOL
    fbs = np.array([fb, fb + 9, fb + 30, fb + 50])
    fes = fbs + np.array([8, 16, 5, 22])
    cn = np.arange(10, 14, dtype=np.uint64)
    c, d = bulk.presync_windows(0.0, fbs, fes, 0.005, 0.04, call_nos=cn)
    assert np.array_equal((c, d), fbf.presync_windows(0.0, fbs, fes, 0.005, 0.04, call_nos=cn))
    for j in range(len(fbs)):
        o.set_rng(SEED, int(cn[j]))
        co, do = o.PreSync(0.0, int(fbs[j]), int(fes[j]), 0.005, 0.04)
        assert d[j] == do and rel_err(c[j], co) <= TOL
    sb, se = np.array([fb + 2, fb + 40]), np.array([fb + 14, fb + 52])
    cs, ds = bulk.sync_batch(np.array([0.035, 0.04]), sb, se, 0.0, 0.2, call_nos=np.array([20, 21], dtype=np.uint64))
    assert np.array_equal((cs, ds), fbf.sync_batch(np.array([0.035, 0.04]), sb, se, 0.0, 0.2,
                                                  call_nos=np.array([20, 21], dtype=np.uint64)))
    co, do = o.sync_batch(np.array([0.035, 0.04]), sb, se, 0.0, 0.2, call_nos=[20, 21])
    assert rel_err(ds, do) <= TOL and rel_err(cs, co) <= TOL


def test_mixed_widths_narrow_frames_in_the_wide_kernel(mixed):
    """windows of 8 frames, one of 512 rays among them: the SLOTS = 16 kernel serves frames of
    2, 3, 17, 33 rays; the window's cost is the sum of the reference's cells"""
    bulk, fbf, o, w, counts = mixed
    rec = bulk.probe_gyro()[2]
    delays = 0.03 + 0.001 * np.arange(2 * GRID_WARPS)
    for lo in (0, 8, 40):
        fb, fe = int(w.frame_ids[lo]), int(w.frame_ids[lo]) + 8
        assert counts[lo:lo + 8].max() == 512
        cb = bulk.presync_grid(fb, fe, delays, call_no=3)
        _, fco, _ = o.presync_grid(fb, fe, delays, call_no=3, frame_costs=True)
        for d, delay in enumerate(delays):
            want, bound = 0.0, 0.0
            for j in range(8):
                i = lo + j
                P = ref.frame_rows(rec, w.gyro_t0, w.gyro_rate, delay, w, i, int(counts[i]))
                cands = ref.presync_cell(P, ref.rng_task_key(SEED, 1, 3, d, int(w.frame_ids[i])))
                best = min(cands, key=lambda cb_: abs(cb_[0] - fco[d, j]))
                assert ref.cell_ratio(fco[d, j], cands) <= 1.0
                want += best[0]
                bound += best[1]
            assert LOG.add("presync_mixed", ref.ratio(cb[d], want, bound + 8 * ref.EPS * want)) <= 1.0


# ------------------------------------------------------------------------------------------------
# C.3  ties in ts_a


def test_tied_timestamps_bulk_frame_by_frame_and_oracle(rsb, oracle_loader):
    """groups of rays that share ts_a exactly (0.0 and -0.0 among them), scattered over the
    caller's order: the sort's tie-break (caller index) fixes the storage and summation order"""
    w = workload("tiny", frames=70, rays=100, seed=SEED, first_frame=0)
    ts_a = w.ts_a.copy()
    rng = np.random.default_rng(3)
    for i in range(w.n_frames):
        ts_a[i] = np.round(ts_a[i] * 400.0) / 400.0  # 2.5 ms rows: ~5 rays per distinct value
        grp = rng.permutation(w.n_rays)[:12]
        ts_a[i, grp] = ts_a[i, grp[0]]
    ts_a[0, ::5] = 0.0
    ts_a[0, 2::7] = -0.0
    assert np.signbit(ts_a[0]).any()
    n = w.n_rays
    counts = np.full(w.n_frames, n)
    bulk = rsb.SyncProblem(seed=SEED)
    bulk.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
    bulk.set_track_batch(w.frame_ids, counts, ts_a, w.ts_b, w.rays_a, w.rays_b)
    fbf = rsb.SyncProblem(seed=SEED)
    o = oracle_loader.OracleProblem(threads=8, seed=SEED)
    for p in (fbf, o):
        p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
        for i, fid in enumerate(w.frame_ids):
            p.SetTrackResult(int(fid), ts_a[i], w.ts_b[i], w.rays_a[i], w.rays_b[i], n)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    for delays in (0.03 + 0.001 * np.arange(2 * GRID_WARPS), np.array([0.0, 0.037])):
        for simplified in (False, True):
            for p in (bulk, fbf, o):
                p.set_loss_mode(simplified)
            cb = bulk.presync_grid(fb, fe, delays, call_no=1)
            assert np.array_equal(cb, fbf.presync_grid(fb, fe, delays, call_no=1))
            assert np.array_equal(cb, o.presync_grid(fb, fe, delays, call_no=1))
            for fid in (fb, fb + 1, fb + 33):
                c1 = bulk.presync_grid(fid, fid + 1, delays, call_no=1)
                assert np.array_equal(c1, o.presync_grid(fid, fid + 1, delays, call_no=1))
    for p in (bulk, fbf, o):
        p.set_loss_mode(False)
    for fid in (fb, fb + 1):
        assert np.array_equal(bulk.probe_problem_matrix(fid, 0.02, n), o.problem_matrix(fid, 0.02, n))
    sb, se = np.array([fb, fb + 30]), np.array([fb + 12, fb + 45])
    cs, ds = bulk.sync_batch(np.array([0.035, 0.04]), sb, se, 0.0, 0.2, call_nos=np.array([7, 8], dtype=np.uint64))
    co, do = o.sync_batch(np.array([0.035, 0.04]), sb, se, 0.0, 0.2, call_nos=[7, 8])
    assert rel_err(ds, do) <= TOL and rel_err(cs, co) <= TOL


# ------------------------------------------------------------------------------------------------
# C.4  gyro-span edges in the production kernel


@pytest.mark.parametrize("simplified", [False, True], ids=["full", "simplified"])
def test_presync_cells_at_the_gyro_span_edges(rsb, oracle_loader, simplified):
    g, o, w, rec = pair(rsb, oracle_loader, 40)
    mode((g, o), simplified)
    nq = rec.shape[0]
    stage = "presync_edges_simplified" if simplified else "presync_edges"
    for i in range(w.n_frames):
        fid = int(w.frame_ids[i])
        edges = ref.span_edge_delays(w, i, nq)
        # the edge delays alone (unstaged, outside the staged window's reach) and a staged run of
        # 16 delays 0.3 ms apart across the last knot
        for delays in (edges, edges[2] - 0.0024 + 0.0003 * np.arange(2 * GRID_WARPS)):
            cg = g.presync_grid(fid, fid + 1, delays, call_no=9)
            assert np.array_equal(cg, o.presync_grid(fid, fid + 1, delays, call_no=9), equal_nan=True)
            for d, delay in enumerate(delays):
                P = ref.frame_rows(rec, w.gyro_t0, w.gyro_rate, delay, w, i)
                assert np.array_equal(g.probe_problem_matrix(fid, delay, w.n_rays), o.problem_matrix(fid, delay, w.n_rays))
                cands = ref.presync_cell(P, ref.rng_task_key(SEED, 1, 9, d, fid), simplified)
                assert LOG.add(stage, ref.cell_ratio(cg[d], cands)) <= 1.0, (fid, delay)
    mode((g, o), False)


# ------------------------------------------------------------------------------------------------
# C.5  degenerate frames


def test_duplicated_ray_gives_the_reference_zero_hypothesis(rsb, oracle_loader):
    """a frame in which a ray is set twice, at the pair the estimator draws first: the reference's
    cross product of the two equal rows is exactly 0, that hypothesis' quartile 0 wins, and
    r = P.M k / |M| = 0 * inf is NaN -- the reference's panic "pre-sync: non-finite r".  The engine
    and the oracle give the same NaN cell and the same error."""
    w = workload("tiny", frames=2, rays=40, seed=SEED)
    fid, n = int(w.frame_ids[0]), w.n_rays
    key = ref.rng_task_key(SEED, 1, 4, 0, fid)
    a, b = ref.draws(key, 20, n)[0]
    ts_a, ts_b, ra, rb = w.ts_a[0].copy(), w.ts_b[0].copy(), w.rays_a[0].copy(), w.rays_b[0].copy()
    ts_a[b], ts_b[b], ra[b], rb[b] = ts_a[a], ts_b[a], ra[a], rb[a]
    g, o = rsb.SyncProblem(seed=SEED), oracle_loader.OracleProblem(threads=2, seed=SEED)
    for p in (g, o):
        p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
        p.SetTrackResult(fid, ts_a, ts_b, ra, rb, n)
    P = ref.rows(g.probe_gyro()[2], w.gyro_t0, w.gyro_rate, 0.0, ts_a, ts_b, ra, rb)
    assert np.isnan(ref.presync_cell(P, key)[0][0])
    delays = np.array([0.0, 0.01])
    cg, fl = g.presync_grid(fid, fid + 1, delays, call_no=4, return_flags=True)
    co, _, flo = o.presync_grid(fid, fid + 1, delays, call_no=4, frame_costs=True)
    assert np.isnan(cg[0]) and np.isnan(co[0]) and fl != 0 and flo != 0
    assert cg[1] == co[1]
    mg, kg = g.probe_guess_motion(fid, 0.0, 20, 1, 4, 0)
    assert np.array_equal(mg, np.zeros(3)) and kg == 1000.0
    errs = []
    for p, E in ((g, rsb.RsSyncError), (o, oracle_loader.OracleError)):
        p.set_rng(SEED, 4)
        with pytest.raises(E) as e:
            p.PreSync(0.0, fid, fid + 1, 0.005, 0.02)
        errs.append((e.value.code, e.value.message))
    assert errs[0] == errs[1] and errs[0][1] == "pre-sync: non-finite r"


def test_frame_ids_that_reach_the_rng_key(rsb, oracle_loader):
    """negative frame ids and ids above 2^31 enter the RNG key as 64-bit values"""
    w = workload("tiny", frames=4, rays=65, seed=SEED)
    ids = [-(2 ** 40), -5, -1, 2 ** 31 + 3, 2 ** 40 + 7]
    g, o = rsb.SyncProblem(seed=SEED), oracle_loader.OracleProblem(threads=2, seed=SEED)
    rec = None
    for p in (g, o):
        p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
        for j, fid in enumerate(ids):
            i = j % w.n_frames
            p.SetTrackResult(fid, w.ts_a[i], w.ts_b[i], w.rays_a[i], w.rays_b[i], w.n_rays)
    rec = g.probe_gyro()[2]
    delays = np.array([0.0, 0.02, 0.037])
    for j, fid in enumerate(ids):
        cg = g.presync_grid(fid, fid + 1, delays, call_no=2)
        assert np.array_equal(cg, o.presync_grid(fid, fid + 1, delays, call_no=2))
        for d, delay in enumerate(delays):
            P = ref.frame_rows(rec, w.gyro_t0, w.gyro_rate, delay, w, j % w.n_frames)
            cands = ref.presync_cell(P, ref.rng_task_key(SEED, 1, 2, d, fid))
            assert LOG.add("presync_ids", ref.cell_ratio(cg[d], cands)) <= 1.0
    lo, hi = -(2 ** 41), 2 ** 41
    assert rel_err(g.presync_grid(lo, hi, delays, call_no=2), o.presync_grid(lo, hi, delays, call_no=2)) <= TOL
    for p in (g, o):
        p.set_rng(SEED, 3)
    sg = g.Sync(0.035, -5, 2 ** 31 + 3, 0.0, 0.2)
    so = o.Sync(0.035, -5, 2 ** 31 + 3, 0.0, 0.2)
    assert rel_err(sg[1], so[1]) <= TOL and rel_err(sg[0], so[0]) <= TOL
