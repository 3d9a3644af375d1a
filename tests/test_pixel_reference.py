"""The pixel -> ray reference (tests/pixel_reference.py) pinned on its own, on the CPU: closed forms, a round
trip through the forward lens model, agreement with synth.undistort, the reference's quirks, the storage
layout, and that its bound is tight enough to see the derivative coefficient 8 k4 become 9 k4."""
import importlib

import numpy as np

import pixel_reference as pr
from conftest import workload
from plain_reference import LD

synth = importlib.import_module("rs-sync_b200.synth")
HERO6 = pr.Lens(*synth.LENS)
EQUIDISTANT = pr.Lens(synth.READOUT, 900.0, 1150.0, 1250.5, 1100.25, 0.0, 0.0, 0.0, 0.0)
STRONG = pr.Lens(synth.READOUT, 600.0, 600.0, 1355.0, 1020.0, -0.3, 0.1, -0.02, 0.01)
CORNERS = np.array([[0.0, 0.0], [synth.WIDTH - 1.0, 0.0], [0.0, synth.HEIGHT - 1.0],
                    [synth.WIDTH - 1.0, synth.HEIGHT - 1.0], [0.0, 1000.0], [1355.0, 0.0]])


def _grid(lo=-150.0, step=97.0):
    xs = np.arange(lo, synth.WIDTH - lo, step)
    ys = np.arange(lo, synth.HEIGHT - lo, step)
    return np.array([(x, y) for y in ys for x in xs])


def test_equidistant_lens_closed_form():
    """k = 0: theta = theta_d, ray (sin theta_d x_ / theta_d, sin theta_d y_ / theta_d, cos theta_d)"""
    L = EQUIDISTANT
    pts = _grid()
    x_ = (pts[:, 0] - L.cx) / L.fx
    y_ = (pts[:, 1] - L.cy) / L.fy
    td = np.sqrt(x_ * x_ + y_ * y_)
    keep = (td > 1e-6) & (td < np.pi / 2 - 1e-3)
    assert keep.sum() > 500
    pts, x_, y_, td = pts[keep], x_[keep].astype(LD), y_[keep].astype(LD), td[keep].astype(LD)
    u = pr.Undistorted(pts, L)
    assert u.converged.all() and not u.root_missing.any()
    want = np.stack([np.sin(td) * x_ / td, np.sin(td) * y_ / td, np.cos(td)], axis=-1)
    assert np.max(pr.angle(want, u.ray) / u.bound) <= 1.0


def test_round_trip_through_the_forward_model():
    """long-double rays -> synth.ray_to_pixel evaluated in long double -> float64 pixels -> the reference"""
    rng = np.random.default_rng(4)
    th = LD(1.25) * np.sqrt(rng.random(2000)).astype(LD)
    ph = (2 * np.pi * rng.random(2000)).astype(LD)
    rays = np.stack([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)], axis=-1)
    px, py = synth.ray_to_pixel(rays)
    assert px.dtype == LD
    u = pr.Undistorted(np.stack([px, py], axis=-1).astype(np.float64), HERO6)
    assert u.converged.all() and not u.root_missing.any()
    assert np.max(pr.angle(rays, u.ray) / u.bound) <= 1.0


def test_agrees_with_synth_undistort():
    """wherever the raw-pixel check (core_testcode.cpp:64) does not apply; where it does they differ"""
    w = workload("tiny", rays=130)
    pts = np.concatenate([w.px_a.reshape(-1, 2), w.px_b.reshape(-1, 2), _grid(-400.0, 131.0),
                          [[1.0, 0.0], [0.0, 1e-6], [HERO6.cx, HERO6.cy]]])
    u = pr.Undistorted(pts, HERO6)
    assert not u.axis.any()
    got = synth.pixel_to_ray(pts[:, 0], pts[:, 1])
    assert np.max(pr.angle(got, u.ray) / u.bound) <= 1.0
    at_origin = pr.Undistorted([[0.0, 0.0]], HERO6)
    assert at_origin.axis[0] and pr.angle(synth.pixel_to_ray(np.zeros(1), np.zeros(1)), at_origin.ray)[0] > 1.0


def test_quirks():
    L = HERO6
    u = pr.Undistorted([[0.0, 0.0], [1e-9, 0.0], [L.cx, L.cy], [L.cx + 5e-10 * L.fx, L.cy],
                        [L.cx, L.cy + 1e-7 * L.fy]], L)
    axis = np.array([0.0, 0.0, 1.0])
    # (0, 0) and (1e-9, 0): the raw-pixel check returns the optical axis
    assert list(u.axis) == [True, True, False, False, False]
    assert np.array_equal(u.ray[:3].astype(np.float64), np.tile(axis, (3, 1)))
    # the principal point: Newton walks to 0 and halves back into (0, pi/2); x_ = y_ = 0 gives the axis
    assert u.theta_d[2] == 0.0 and u.halvings[2] > 0 and 0.0 < u.theta[2] < np.pi / 2
    # theta_d = 5e-10 takes the 1 / cos branch, 1e-7 the tan one; both converge
    assert list(u.small) == [False, False, True, True, False]
    assert u.converged[3] and u.converged[4]
    assert np.max(pr.angle(u.ray[3:], [[5e-10, 0.0, 1.0], [0.0, 1e-7, 1.0]]) / u.bound[3:]) <= 1.0


def test_far_points_and_strong_lens_replay():
    """outside the image circle and on a strong lens the 9 Newton steps do not converge: the replayed theta
    is the answer, after dozens of halvings"""
    u = pr.Undistorted([[-3000.0, 5000.0], [1e5, 1e5]], HERO6)
    assert not u.converged.any() and (u.halvings >= 50).all()
    s = pr.Undistorted(CORNERS, STRONG)
    assert not s.converged.any() and (s.halvings >= 50).all()
    assert np.all(np.isfinite(s.ray.astype(np.float64)))


def test_nine_k4_is_detected():
    """the exact derivative coefficient 9 k4 in place of the reference's 8 k4 moves the replayed rays of
    the strong lens's corners by more than 1e6 bound units, and the Hero6 corners (converged) not at all"""
    ref, mut = pr.Undistorted(CORNERS, STRONG), pr.Undistorted(CORNERS, STRONG, k4_coef=9.0)
    moved = pr.angle(ref.ray, mut.ray) / ref.bound
    assert np.min(moved[1:]) > 1e6, moved
    h, h9 = pr.Undistorted(CORNERS, HERO6), pr.Undistorted(CORNERS, HERO6, k4_coef=9.0)
    assert h.converged[1:].all() and np.max(pr.angle(h.ray, h9.ray) / h.bound) <= 1.0


def test_storage_layout():
    """sorted by (ts_a, caller index); tiles [8 fields][32 lanes]; orig / pos; padding lanes; bounds"""
    rng = np.random.default_rng(2)
    n = 45
    pa = np.column_stack([rng.uniform(0, 2000, n), rng.choice([0.0, 400.0, 1800.0], n)])  # tied rows
    pb = pa + rng.normal(0, 2, (n, 2))
    f = pr.Frame(pa, pb, 1.5, 1.6, HERO6, synth.HEIGHT)
    assert f.tiles.shape == (2, 8, 32)
    flat = f.tiles.transpose(1, 0, 2).reshape(8, 64)
    keys = list(zip(flat[0, :n], f.orig[:n]))
    assert keys == sorted(keys) and len(set(f.ts_a)) == 3
    assert np.array_equal(f.pos[f.orig[:n]], np.arange(n)) and np.array_equal(f.orig[n:], np.arange(n, 64))
    assert np.array_equal(f.pos[n:], np.arange(n, 64))
    assert np.array_equal(flat[1, :n], f.ts_b[f.orig[:n]])
    assert np.array_equal(flat[2:5, :n].T, f.und_a.ray.astype(np.float64)[f.orig[:n]])
    last = f.orig[n - 1]
    assert (flat[0, n:] == f.ts_a[last]).all() and (flat[1, n:] == f.ts_b[last]).all() and not flat[2:, n:].any()
    assert (f.ts_lo, f.ts_hi) == (min(f.ts_a.min(), f.ts_b.min()), max(f.ts_a.max(), f.ts_b.max()))
    assert f.ts_lo == 1.5 and f.ts_a.max() < f.ts_b.max()
    # at readout 0 every ray ties: caller order
    z = f.retimed(pa, pb, 1.5, 1.6, HERO6, synth.HEIGHT, 0.0)
    assert np.array_equal(z.orig[:n], np.arange(n)) and (z.ts_lo, z.ts_hi) == (1.5, 1.6)
    e = pr.Frame(np.zeros((0, 2)), np.zeros((0, 2)), 1.5, 1.6, HERO6, synth.HEIGHT)
    assert e.tiles.shape == (0, 8, 32) and (e.ts_lo, e.ts_hi) == (0.0, 0.0)
