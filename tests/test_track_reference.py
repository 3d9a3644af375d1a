"""The tracker restatement (tests/track_reference.py) and the renderer (tests/render_reference.py) pinned on
their own, on the CPU: the pyramid against cv2.pyrDown, the tracker against cv2's Lucas-Kanade on rendered
frames with known correspondences, and the renderer's correspondences through the lens model."""
import importlib

import numpy as np
import pytest

import render_reference as rr
import track_reference as tr

cv2 = pytest.importorskip("cv2")
rsb = importlib.import_module("rs-sync_b200")


@pytest.mark.parametrize("shape", [(240, 320), (241, 323), (7, 5), (1014, 1352)])
def test_pyramid_matches_cv2_pyrdown(shape):
    rng = np.random.default_rng(shape)
    img = rng.integers(0, 256, shape).astype(np.float32)
    for lvl in range(3):
        ref = cv2.pyrDown(img)
        ours = tr.pyr_down(img)
        assert ours.shape == ref.shape == ((img.shape[0] + 1) // 2, (img.shape[1] + 1) // 2)
        assert np.max(np.abs(ours - ref) / np.maximum(np.abs(ref), 1.0)) <= 1e-5
        img = ref
        if min(img.shape) < 3:
            break


@pytest.fixture(scope="module")
def small_clip():
    clip = rr.Clip(320, 240, 4, delay=0.02)
    return clip, clip.render_all()


def test_renderer_correspondences_round_trip(small_clip):
    clip, _ = small_clip
    pts = rsb.grid_points(clip.width, clip.height, 25)
    r = clip.pixel_to_ray(pts[:, 0], pts[:, 1])
    x, y = clip.ray_to_pixel(r)
    assert np.max(np.hypot(x - pts[:, 0], y - pts[:, 1])) < 1e-6
    for j in range(clip.n_images - 1):
        b = clip.true_b(j, pts)
        # the fixed point: the world direction seen at b, at b's row time, is the one seen at a
        wa = clip.world(j, pts[:, 0], pts[:, 1])
        wb = clip.world(j + 1, b[:, 0], b[:, 1])
        assert np.max(np.linalg.norm(wa - wb, axis=1)) < 1e-9
        assert np.max(np.hypot(*(b - pts).T)) > 0.5  # the camera moves


def _errors(tracked, status, truth):
    e = np.hypot(*(tracked - truth).T)
    return e[status]


def test_restatement_no_worse_than_cv2_lk(small_clip):
    clip, imgs = small_clip
    pts = rsb.grid_points(clip.width, clip.height, 20)
    inside = (pts[:, 0] >= 15) & (pts[:, 0] <= clip.width - 16) & (pts[:, 1] >= 15) & (pts[:, 1] <= clip.height - 16)
    pts = pts[inside]
    ours, theirs = [], []
    for j in range(clip.n_images - 1):
        truth = clip.true_b(j, pts)
        res = tr.track(imgs[j], imgs[j + 1], pts)
        p1, st, _ = cv2.calcOpticalFlowPyrLK(imgs[j], imgs[j + 1], pts.astype(np.float32).reshape(-1, 1, 2), None,
                                             winSize=(21, 21), maxLevel=2,
                                             criteria=(cv2.TERM_CRITERIA_COUNT | cv2.TERM_CRITERIA_EPS, 30, 0.01))
        both = res["status"] & (st.ravel() == 1)
        ours.append(_errors(res["tracked"], both, truth))
        theirs.append(_errors(p1.reshape(-1, 2).astype(np.float64), both, truth))
        assert res["status"].mean() > 0.95
    ours, theirs = np.concatenate(ours), np.concatenate(theirs)
    for q in (50, 90):
        assert np.percentile(ours, q) <= np.percentile(theirs, q) + 0.02, (q, np.percentile(ours, q),
                                                                           np.percentile(theirs, q))


def test_restatement_statuses():
    """lost: starts outside, ends outside, flat (eigenvalue) windows; kept: a textured interior point"""
    rng = np.random.default_rng(3)
    a = rng.integers(0, 256, (64, 64)).astype(np.float64)
    a = tr.pyr_down(np.kron(a, np.ones((2, 2))))  # smooth enough to track
    b = np.roll(a, 1, axis=1)
    flat = np.full((64, 64), 7.0)
    pts = np.array([[30.0, 30.0], [-0.5, 10.0], [63.0, 63.0], [np.nan, 3.0], [63.5, 2.0]])
    res = tr.track(a, b, pts, tr.Params(levels=2, window=9))
    assert res["status"].tolist() == [True, False, False, False, False]
    assert abs(res["tracked"][0, 0] - 31.0) < 0.05 and abs(res["tracked"][0, 1] - 30.0) < 0.05
    res = tr.track(flat, flat, pts[:1], tr.Params(levels=2, window=9))
    assert not res["status"][0]


def test_grid_points_is_centred():
    g = rsb.grid_points(2704, 2028, 200)
    assert g.shape == (14 * 11, 2)
    assert np.allclose(g[0], [(2703 - 2600) / 2, (2027 - 2000) / 2])
    assert np.allclose(g[0] + g[-1], [2703, 2027])
    assert np.all(np.diff(g[:14, 0]) == 200)
