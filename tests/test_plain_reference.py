"""The CPU oracle against an independent long-double restatement of the reference's math
(tests/plain_reference.py), on every ray count that crosses a SLOTS boundary of the engine's
kernels or a quartile-rank edge, and at the edges of the gyro span.

Engine and oracle share one arithmetic contract, so their bit-for-bit agreement cannot show that
either computes the reference's formulas: a quartile rank, a constant or an order wrong in the
same way on both sides passes every engine-vs-oracle test.  These tests close that gap for the
oracle; tests/test_gpu_kernel_matrix.py closes it for the kernels.  Values are compared under the
per-value bound of plain_reference (the largest ratio seen per stage is printed, run with -s).
"""
import json
import os

import numpy as np
import pytest

import plain_reference as ref
from conftest import workload

# both sides of every slots_for boundary (2, 4, 6, 7, 8, 12, 16 slots of 32 rays) and the
# quartile-rank edges n // 4 = 0, 1
RAY_COUNTS = [2, 3, 4, 5, 31, 32, 33, 64, 65, 128, 129, 192, 193, 224, 225, 256, 257, 384, 385, 512]
SEED = 29
LOG = ref.RatioLog()


def _oracle(oracle_loader, w, seed=SEED, simplified=False):
    o = oracle_loader.OracleProblem(threads=4, seed=seed).load(w)
    o.set_loss_mode(simplified)
    return o


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("\nplain reference vs oracle, largest bound ratio per stage:", LOG.report())


def test_rng_restatement_reproduces_golden_draws():
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "rng_draws.json")))
    got = [ref.rng_index(ref.rng_task_key(100, 1, 0, d, 3900), it, k, 200)
           for d in (0, 7) for it in (0, 19) for k in (0, 1)]
    assert got == g["draws"]


def test_rng_restatement_matches_oracle(oracle_loader):
    L = oracle_loader.lib()
    for seed, stream, call, off, fid in ((1, 1, 0, 0, 0), (7, 3, 5, 99, -3), (2 ** 63, 2, 2 ** 40, 2 ** 33, 2 ** 40 + 7)):
        for it, k, n in ((0, 0, 2), (5, 3, 3), (199, 1, 512), (17, 0, 7)):
            want = L.orc_rng_index(seed, stream, call, off, fid, it, k, n)
            assert ref.rng_index(ref.rng_task_key(seed, stream, call, off, fid), it, k, n) == want


@pytest.mark.parametrize("nq", [2, 3, 5, 64, 2001])
def test_spline_records_against_scipy(oracle_loader, nq):
    """the oracle's {y, b, c, d} records are SciPy's natural CubicSpline at every knot, the last
    record's b (the slope the right-hand extrapolation uses) included"""
    from scipy.interpolate import CubicSpline
    rng = np.random.default_rng(nq)
    q = rng.normal(size=(nq, 4))
    o = oracle_loader.OracleProblem()
    o.SetGyroQuaternions(q, nq, 1000.0, 0.0)
    rec = o.spline()
    cs = CubicSpline(np.arange(nq, dtype=np.float64), q, bc_type="natural")
    scale = max(1.0, float(np.max(np.abs(q))))
    assert np.max(np.abs(rec[:, 0:4] - q)) == 0.0
    assert np.max(np.abs(rec[:-1, 4:8] - cs.c[2].reshape(nq - 1, 4))) <= 1e-13 * scale
    assert np.max(np.abs(rec[:-1, 8:12] - cs.c[1].reshape(nq - 1, 4))) <= 1e-13 * scale
    assert np.max(np.abs(rec[:-1, 12:16] - cs.c[0].reshape(nq - 1, 4))) <= 1e-13 * scale
    assert np.max(np.abs(rec[-1, 4:8] - cs(nq - 1.0, 1))) <= 1e-13 * scale
    assert np.max(np.abs(rec[-1, 8:16])) <= 1e-13 * scale


def test_spline_evaluation_at_the_span_edges(oracle_loader, w_tiny):
    """left of the first knot (linear), on exact integers, in [n - 1, n) and at x >= n (the
    reference's sawtooth: h = x - min(floor(x), n) restarts at n)"""
    o = _oracle(oracle_loader, w_tiny)
    rec = o.spline()
    n = rec.shape[0]
    x = np.array([-3.5, -1.0, -1e-9, -0.0, 0.0, 1e-12, 0.5, 1.0, 2.0, n / 2.0, n - 2.0, n - 1.5, n - 1.0,
                  n - 1.0 + 1e-9, n - 0.5, n - 1e-9, float(n), n + 1e-9, n + 0.25, n + 0.999, n + 1.0, n + 7.5])
    got = o.spline_eval(x)
    want = ref.spline_eval(rec, x).astype(np.float64)
    h = np.abs(x - np.clip(np.floor(x), 0, n))
    bound = ref.E * (1 + h) ** 3 * float(np.max(np.abs(rec)))
    assert LOG.add("spline", ref.ratio(got, want, bound[:, None])) <= 1.0
    # the sawtooth: just below n the last record is evaluated at h ~ 1, at n at h = 0
    at_n = int(np.flatnonzero(x == n)[0])
    assert np.array_equal(got[at_n], rec[-1, 0:4])
    assert np.max(np.abs(got[at_n - 1] - rec[-1, 0:4])) > 1e3 * ref.E


def _workload(n, frames=3):
    return workload("tiny", frames=frames, rays=n, seed=SEED)


@pytest.mark.parametrize("n", RAY_COUNTS)
def test_oracle_stages_against_plain_reference(oracle_loader, n):
    """rows, the estimator's choice (20 and 200 hypotheses), k, Loss3, Loss5 and its gradient"""
    w = _workload(n)
    o = _oracle(oracle_loader, w)
    rec = o.spline()
    q0, sr = w.gyro_t0, w.gyro_rate
    for i in range(w.n_frames):
        fid = int(w.frame_ids[i])
        for off, delay in enumerate((0.0, 0.037, -0.02)):
            P = ref.frame_rows(rec, q0, sr, delay, w, i)
            Po = o.problem_matrix(fid, delay, n)
            assert LOG.add("rows", ref.ratio(Po, P.astype(np.float64), ref.E)) <= 1.0
            for iters, stream in ((20, 1), (200, 3)):
                key = ref.rng_task_key(SEED, stream, 2, off, fid)
                est = ref.Estimate(P, key, iters)
                m, k = o.guess_motion(fid, delay, iters, stream, 2, off)
                # the chosen hypothesis is one of the reference's near-ties, to the rounding of a row
                d = [ref.ratio(m, est.hyp[t].astype(np.float64), est.dM[t]) for t in est.near]
                assert LOG.add("estimator", min(d)) <= 1.0, (fid, delay, iters, est.near, est.quartile[est.best])
                t = est.near[int(np.argmin(d))]
                _, _, kr, dk = ref.presync_cost(P, est.hyp[t], float(est.dM[t]))
                assert LOG.add("k", ref.ratio(k, kr, dk)) <= 1.0
                l3, b3 = ref.loss3(P, m, k)
                assert LOG.add("loss3", ref.ratio(o.loss3(fid, delay, m, k), l3, b3)) <= 1.0
                l5, g5, b5, bg = ref.loss5(P, m, k)
                l5o, g5o = o.loss5(fid, delay, m, k)
                assert LOG.add("loss5", ref.ratio(l5o, l5, b5)) <= 1.0
                assert LOG.add("gradient", ref.ratio(g5o, g5, bg)) <= 1.0


@pytest.mark.parametrize("simplified", [False, True], ids=["full", "simplified"])
@pytest.mark.parametrize("n", RAY_COUNTS)
def test_oracle_presync_cells_against_plain_reference(oracle_loader, n, simplified):
    """every (delay, frame) cost of a PreSync grid"""
    w = _workload(n)
    o = _oracle(oracle_loader, w, simplified=simplified)
    rec = o.spline()
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    delays = np.array([-0.03, 0.0, 0.021, 0.037, 0.05])
    costs, fc, flags = o.presync_grid(fb, fe, delays, call_no=3, offset_index_base=11, frame_costs=True)
    assert flags == 0
    for d, delay in enumerate(delays):
        for i in range(w.n_frames):
            P = ref.frame_rows(rec, w.gyro_t0, w.gyro_rate, delay, w, i)
            key = ref.rng_task_key(SEED, 1, 3, 11 + d, int(w.frame_ids[i]))
            cands = ref.presync_cell(P, key, simplified)
            assert LOG.add("presync_simplified" if simplified else "presync", ref.cell_ratio(fc[d, i], cands)) <= 1.0


@pytest.mark.parametrize("simplified", [False, True], ids=["full", "simplified"])
def test_oracle_cells_at_the_gyro_span_edges(oracle_loader, simplified):
    w = _workload(40, frames=2)
    o = _oracle(oracle_loader, w, simplified=simplified)
    rec = o.spline()
    nq = rec.shape[0]
    fid = int(w.frame_ids[1])
    delays = ref.span_edge_delays(w, 1, nq)
    costs, fc, flags = o.presync_grid(fid, fid + 1, delays, call_no=1, frame_costs=True)
    for d, delay in enumerate(delays):
        P = ref.frame_rows(rec, w.gyro_t0, w.gyro_rate, delay, w, 1)
        assert LOG.add("rows_edges", ref.ratio(o.problem_matrix(fid, delay, w.n_rays), P.astype(np.float64), ref.E)) <= 1.0
        cands = ref.presync_cell(P, ref.rng_task_key(SEED, 1, 1, d, fid), simplified)
        assert LOG.add("presync_edges", ref.cell_ratio(fc[d, 0], cands)) <= 1.0


def test_oracle_duplicated_ray_gives_the_reference_zero_hypothesis(oracle_loader):
    """a ray set twice, at the pair the estimator draws first: the reference's cross product of the
    two equal rows is exactly 0, that hypothesis wins with quartile 0, and r = 0 * inf is NaN --
    the reference's panic "pre-sync: non-finite r", which the oracle reports too"""
    w = _workload(40, frames=1)
    fid, n = int(w.frame_ids[0]), w.n_rays
    key = ref.rng_task_key(SEED, 1, 4, 0, fid)
    a, b = ref.draws(key, 20, n)[0]
    ts_a, ts_b, ra, rb = w.ts_a[0].copy(), w.ts_b[0].copy(), w.rays_a[0].copy(), w.rays_b[0].copy()
    ts_a[b], ts_b[b], ra[b], rb[b] = ts_a[a], ts_b[a], ra[a], rb[a]
    o = oracle_loader.OracleProblem(seed=SEED)
    o.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
    o.SetTrackResult(fid, ts_a, ts_b, ra, rb, n)
    P = ref.rows(o.spline(), w.gyro_t0, w.gyro_rate, 0.0, ts_a, ts_b, ra, rb)
    assert np.isnan(ref.presync_cell(P, key)[0][0])
    m, k = o.guess_motion(fid, 0.0, 20, 1, 4, 0)
    assert np.array_equal(m, np.zeros(3)) and k == 1000.0
    costs, fc, flags = o.presync_grid(fid, fid + 1, np.array([0.0, 0.01]), call_no=4, frame_costs=True)
    assert np.isnan(costs[0]) and flags & 4 and np.isfinite(costs[1])
    o.set_rng(SEED, 4)
    with pytest.raises(oracle_loader.OracleError) as e:
        o.PreSync(0.0, fid, fid + 1, 0.005, 0.02)
    assert e.value.message == "pre-sync: non-finite r"
