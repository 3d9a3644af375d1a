"""Gyro axis mappings as 3x3 matrices (rssync_integrate_gyro_matrix, the mapping arithmetic of
rs-sync_b200/csrc/gyro_scan.h), the helpers around them (orientation_matrix, rotations_about,
estimate_angle), the sharded rotation search on the oracle, and the mount-rotation recovery experiment on
the CPU oracle.  The oracle side of the matrix mapping is tests/rotation_reference.py (numpy restatement of
the mapping rule, then the oracle's own integration).

The recovery experiment gives a C1-shaped scene a gyro logged in a frame tilted by a known angle,
gyro_imu = omega @ R_true (so the mapping that undoes it is R_true itself), and sweeps candidate rotations
about the tilt axis: 0 .. 50 degrees in 5-degree steps, then +-5 degrees around the coarse argmin in
1-degree steps.  The cost of a candidate is its PreSync minimum, with the RNG call numbers a fresh problem
gives (0, 1, ... over both sweeps).  The PreSync minimum is V-shaped in the angle rather than parabolic, so
the coarse sweep's parabola is only good to ~2 degrees; the fine sweep's vertex is the estimate.  The
largest error it measures pins the tolerance of the GPU recovery test (tests/test_gpu_rotation_search.py),
which runs the same settings through the engine."""
import importlib
import os
import sys

import numpy as np
import pytest

import rotation_reference as ref
from conftest import ROOT, workload

# the recovery settings, shared with the GPU test
INITIAL, STEP, RADIUS = 0.037, 0.0005, 0.012
COARSE_DEG = np.arange(0.0, 50.1, 5.0)
# (seed, axis, true tilt in degrees).  |estimate - truth| the oracle gives: 0.03, 0.39 and 0.68 degrees;
# the engine's costs differ from the oracle's by rounding, hence some margin
RECOVERY_CASES = [(1, "x", 25.0), (2, "y", 18.0), (3, "x", 32.0)]
RECOVERY_TOL_DEG = 1.0


def _pkg():
    return importlib.import_module("rs-sync_b200")


def _u64(a):
    return np.ascontiguousarray(a).view(np.uint64)


def _random_rotations(rng, n):
    out = []
    for _ in range(n):
        q, r = np.linalg.qr(rng.normal(size=(3, 3)))
        q = q * np.sign(np.diag(r))
        if np.linalg.det(q) < 0:
            q[:, 0] = -q[:, 0]
        out.append(q)
    return out


def _gyro_track(n, seed):
    rng = np.random.default_rng(seed)
    ts = np.sort(10.0 + np.arange(n) / 800.0 + rng.uniform(-2e-4, 2e-4, n))
    g = rng.normal(scale=2.0, size=(n, 3))
    g[n // 3:n // 3 + 7] = 0.0  # theta^2 = 0 under any matrix: the quat_from_aa branch of quat.cpp:13-16
    return ts, g


def test_matrix_integration_equals_the_oracle(rsb, oracle_loader):
    n = 3 * 512 + 211  # more than 3 scan blocks
    ts, g = _gyro_track(n, 4)
    rng = np.random.default_rng(11)
    mats = _random_rotations(rng, 5) + [
        np.array([[1.3, -0.2, 0.05], [0.0, 0.9, 0.4], [-0.7, 0.0, 1.1]]),  # not orthogonal, with zeros
        np.diag([1.02, 0.97, 1.0]),                                            # a gain error
        np.zeros((3, 3)),                                                      # every increment the identity
        -np.eye(3),
    ]
    for m in mats:
        a = rsb.integrate_gyro(ts, g, rotation=m)
        b = ref.integrate_gyro(oracle_loader, ts, g, m)
        assert np.array_equal(_u64(a), _u64(b)), m
    assert np.array_equal(rsb.integrate_gyro(ts, g, rotation=np.zeros((3, 3))), np.tile([1.0, 0, 0, 0], (n, 1)))
    # zero rate: the theta^2 = 0 branch for every sample
    z = rsb.integrate_gyro(ts[:5], np.zeros((5, 3)), rotation=mats[0])
    assert np.array_equal(z, np.tile([1.0, 0, 0, 0], (5, 1)))


def test_identity_equals_no_mapping(rsb, oracle_loader):
    ts, g = _gyro_track(1500, 5)
    a = rsb.integrate_gyro(ts, g)
    for q in (rsb.integrate_gyro(ts, g, rotation=np.eye(3)), ref.integrate_gyro(oracle_loader, ts, g, np.eye(3)),
              oracle_loader.integrate_gyro(ts, g)):
        assert np.array_equal(_u64(a), _u64(q))


def test_every_orientation_string_is_its_matrix(rsb, oracle_loader, synth_mod):
    """the zero-coefficient rule makes a signed permutation matrix reproduce the string's bits: signed
    zeros, and a NaN on an axis the mapping does not read (which must not reach the result)"""
    ts, g = _gyro_track(1200, 6)
    g[10:20] = 0.0
    g[20:30] = -0.0
    g[30:40, 0] = -0.0
    g[40:50, 1] = 0.0
    g[600, 2] = np.nan  # axis z of one sample
    for s in synth_mod.ORIENTATIONS:
        m = rsb.orientation_matrix(s)
        want = rsb.integrate_gyro(ts, g, orientation=s)
        for got in (rsb.integrate_gyro(ts, g, rotation=m), ref.integrate_gyro(oracle_loader, ts, g, m),
                    oracle_loader.integrate_gyro(ts, g, s)):
            assert np.array_equal(_u64(want), _u64(got)), s
        assert np.isnan(want[600:]).all() == ("z" in s.lower())
    assert np.array_equal(rsb.orientation_matrix(None), np.eye(3))


def test_orientation_matrix_and_rotations_about(rsb, synth_mod, w_tiny):
    om = w_tiny.omega
    for s in synth_mod.ORIENTATIONS:
        assert np.array_equal(om @ rsb.orientation_matrix(s).T, synth_mod.orient_omega(om, s)), s
    th = np.linspace(-3.0, 3.0, 13)
    for axis in "xyz":
        R = rsb.rotations_about(axis, th)
        assert R.shape == (13, 3, 3)
        for r in R:
            assert np.max(np.abs(r @ r.T - np.eye(3))) <= 1e-15 * 4
            assert np.linalg.det(r) == pytest.approx(1.0, abs=1e-15 * 4)
        back = rsb.rotations_about(axis, -th)
        for r, b in zip(R, back):
            assert np.max(np.abs(b @ r - np.eye(3))) <= 1e-15 * 2
        k = "xyz".index(axis)
        assert np.array_equal(R[:, k, k], np.ones(13)) and np.array_equal(R[:, k, [j for j in range(3) if j != k]],
                                                                          np.zeros((13, 2)))
    # right-handed: a quarter turn about z takes x to y, about x takes y to z, about y takes z to x
    quarter = np.pi / 2
    assert np.allclose(rsb.rotations_about("z", [quarter])[0] @ [1, 0, 0], [0, 1, 0], atol=1e-16)
    assert np.allclose(rsb.rotations_about("x", [quarter])[0] @ [0, 1, 0], [0, 0, 1], atol=1e-16)
    assert np.allclose(rsb.rotations_about("y", [quarter])[0] @ [0, 0, 1], [1, 0, 0], atol=1e-16)


def test_rejections(rsb, oracle_loader):
    ts, g = _gyro_track(20, 7)
    for bad in (np.nan, np.inf, -np.inf):
        m = np.eye(3)
        m[1, 2] = bad
        with pytest.raises(rsb.RsSyncError) as e:
            rsb.integrate_gyro(ts, g, rotation=m)
        assert e.value.code == rsb.E_INVALID
        with pytest.raises(ValueError, match="non-finite"):
            ref.map_gyro(m, g)
    for shape in ((3,), (9,), (2, 3), (3, 4), (1, 3, 3)):
        with pytest.raises(ValueError, match="3x3"):
            rsb.integrate_gyro(ts, g, rotation=np.ones(shape))
        with pytest.raises(ValueError, match="3x3"):
            ref.map_gyro(np.ones(shape), g)
    with pytest.raises(ValueError, match="not both"):
        rsb.integrate_gyro(ts, g, orientation="XYZ", rotation=np.eye(3))
    for bad in ("XY", "XYZW", "XYQ", "", 3):
        with pytest.raises(ValueError, match="malformed"):
            rsb.orientation_matrix(bad)
    with pytest.raises(ValueError, match="axis"):
        rsb.rotations_about("w", [0.1])


def test_estimate_angle_exact_parabolas():
    est = _pkg().estimate_angle
    deg = np.deg2rad(np.arange(0.0, 50.1, 5.0))
    for vertex, a, c0 in [(0.4, 3.0e3, 1500.0), (0.01, 1.0, 0.0), (0.85, 5.0e4, -7.0), (-0.2, 2.0, 1.0)]:
        x = deg if vertex >= 0 else deg - 0.5
        assert est(x, a * (x - vertex) ** 2 + c0) == pytest.approx(vertex, abs=1e-12)
    x = np.array([0.3, 0.1, 0.2])
    assert est(x, (x - 0.15) ** 2) == pytest.approx(0.15, abs=1e-14)


def test_estimate_angle_rejections():
    est = _pkg().estimate_angle
    x = np.deg2rad(np.arange(0.0, 50.1, 5.0))
    with pytest.raises(ValueError, match="not convex"):
        est(x, -(x - 0.4) ** 2)
    with pytest.raises(ValueError, match="not convex"):
        est(x, 2.0 * x + 1.0)
    with pytest.raises(ValueError, match="outside the candidate angles"):
        est(x, (x - 1.5) ** 2)
    with pytest.raises(ValueError, match="3 distinct angles"):
        est([0.1, 0.1, 0.2], [1.0, 1.0, 2.0])
    with pytest.raises(ValueError, match="angles but"):
        est(x, x[:-1])
    with pytest.raises(ValueError, match="angles and costs must be finite"):
        est(x, np.where(x > 0.4, np.nan, x))


# ---- the sharded rotation search (variant k on rank k % world) on the oracle ---------------------------
def _scene():
    synth = importlib.import_module("rs-sync_b200.synth")
    w = synth.make_workload("tiny", first_frame=200)
    ts = w.gyro_t0 + np.arange(w.quats.shape[0]) / w.gyro_rate
    rots = list(_pkg().rotations_about("x", np.deg2rad([0.0, 10.0, -20.0]))) + [np.diag([1.0, 1.0, 1.05])]
    return w, ts, rots


def _worker(rank, world, port, q):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sharded = importlib.import_module("rs-sync_b200.sharded")
    from oracle import loader
    import rotation_reference
    w, ts, rots = _scene()
    o = loader.OracleProblem(threads=1, seed=100).load(w)

    def batch(pr, ms, call_nos):
        cs, ds = [], []
        for m, cn in zip(ms, call_nos):
            pr.set_rng(100, int(cn))
            c_, d_ = rotation_reference.rotation_search(loader, pr, ts, w.omega, [m], 0.0, 200, 212, 0.01, 0.05)
            cs.append(c_[0])
            ds.append(d_[0])
        return np.array(cs), np.array(ds)

    c, d = sharded.orientation_search_sharded(o, None, rots, seed=100, call_no_base=7, rank=rank, world=world,
                                              batch_fn=batch)
    if rank == 0:
        q.put((c, d))
    dist.barrier()
    dist.destroy_process_group()


def test_rotation_search_sharded_world2(oracle_loader):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    c, d = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    w, ts, rots = _scene()
    o = oracle_loader.OracleProblem(threads=2, seed=100).load(w)
    o.set_rng(100, 7)
    wc, wd = ref.rotation_search(oracle_loader, o, ts, w.omega, rots, 0.0, 200, 212, 0.01, 0.05)
    assert np.array_equal(c, wc) and np.array_equal(d, wd)


# ---- recovery of a known mount tilt -------------------------------------------------------------------
def recovery_scene(seed, axis, true_deg):
    """(workload, gyro timestamps, gyro in the tilted frame, frame range)"""
    w = workload("C1", seed=seed, first_frame=200)  # non-negative microsecond timestamps (SURVEY a3)
    ts = w.gyro_t0 + np.arange(w.quats.shape[0]) / w.gyro_rate
    r_true = _pkg().rotations_about(axis, [np.deg2rad(true_deg)])[0]
    return w, ts, w.omega @ r_true, (int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1)


def fine_candidates_deg(coarse_costs):
    """+-5 degrees around the coarse argmin in 1-degree steps, clipped to the coarse range"""
    k = int(np.argmin(coarse_costs))
    lo, hi = max(COARSE_DEG[k] - 5.0, COARSE_DEG[0]), min(COARSE_DEG[k] + 5.0, COARSE_DEG[-1])
    return np.arange(lo, hi + 0.5, 1.0)


def estimate_tilt_deg(search, axis):
    """the coarse-then-fine sweep; search(rotations) -> PreSync minima, called twice in order"""
    rsb = _pkg()
    coarse = search(rsb.rotations_about(axis, np.deg2rad(COARSE_DEG)))
    fine = fine_candidates_deg(coarse)
    costs = search(rsb.rotations_about(axis, np.deg2rad(fine)))
    return float(np.rad2deg(rsb.estimate_angle(np.deg2rad(fine), costs)))


@pytest.mark.parametrize("seed,axis,true_deg", RECOVERY_CASES)
def test_recovery_on_the_oracle(oracle_loader, seed, axis, true_deg):
    w, ts, gyro, (fb, fe) = recovery_scene(seed, axis, true_deg)
    o = oracle_loader.OracleProblem(threads=os.cpu_count() or 1, seed=100).load(w)
    est = estimate_tilt_deg(
        lambda rots: ref.rotation_search(oracle_loader, o, ts, gyro, rots, INITIAL, fb, fe, STEP, RADIUS)[0], axis)
    assert abs(est - true_deg) <= RECOVERY_TOL_DEG, (seed, axis, true_deg, est)
