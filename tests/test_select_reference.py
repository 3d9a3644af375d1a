"""The selection restatement (tests/select_reference.py) pinned on its own, on the CPU: its scores against
cv2.cornerMinEigenVal, known answers of the cell rule, the threshold and the max_points cut, the backward pass
composed from the tracker restatement, and the new C symbols."""
import importlib

import numpy as np
import pytest

import render_reference as rr
import select_reference as sr
import track_reference as tr
from test_abi import declared_symbols

cv2 = pytest.importorskip("cv2")
rsb = importlib.import_module("rs-sync_b200")


def _noise(shape, seed):
    rng = np.random.default_rng(seed)
    return cv2.GaussianBlur(rng.integers(0, 256, shape).astype(np.uint8), (5, 5), 1.2)


@pytest.fixture(scope="module")
def rendered():
    return rr.Clip(320, 240, 1, delay=0.02, seed=2).render(0)


@pytest.mark.parametrize("block", [3, 5, 7])
def test_scores_match_cv2(rendered, block):
    """within 1e-6 of the image's maximum on blurred noise.  On the rendered frames, whose smooth texture has
    strong gradients and weak corners, cv2's box filter (running sums) rounds differently: the difference is
    up to about 100 float32 ulps of the larger eigenvalue, 3.1e-6 of the maximum score, so there the bound is
    5e-6 of the maximum."""
    for img, tol in ((rendered, 5e-6), (_noise((97, 131), block), 1e-6), (_noise((240, 320), 10 + block), 1e-6)):
        ref = cv2.cornerMinEigenVal(img, block, 3)
        ours = sr.scores(img, block)
        assert ours.dtype == np.float32
        err = np.max(np.abs(ours - ref)) / ref.max()
        print(f"block {block}, {img.shape}: max |restatement - cv2| / max score = {err:.3g}")
        assert err <= tol, (block, img.shape, err)


def _squares(shape, squares, value=255):
    img = np.zeros(shape, dtype=np.uint8)
    for x0, y0, side in squares:
        img[y0:y0 + side, x0:x0 + side] = value
    return img


@pytest.mark.parametrize("block", [3, 5, 7])
def test_square_corners(block):
    """bright squares on black: one pick per corner, within 1 px of it for block 3.  On a hard step the
    detector's maximum sits block / 2 - 1 px inside the square along the diagonal (cv2.goodFeaturesToTrack
    picks the same pixels), so the larger blocks are held to that point."""
    sq = [(20, 30, 40), (110, 25, 33), (70, 100, 45)]
    img = _squares((180, 200), sq)
    pts = sr.select(img, sr.Options(cell=16, block=block))["points"]
    inset = block // 2 - 1
    corners = np.array([(x - 0.5 + dx, y - 0.5 + dy) for x, y, s in sq for dx in (0, s) for dy in (0, s)])
    towards = np.array([(1 if dx == 0 else -1, 1 if dy == 0 else -1) for x, y, s in sq for dx in (0, s)
                        for dy in (0, s)])
    d = np.hypot(*(pts[:, None, :] - (corners + inset * towards)[None]).transpose(2, 0, 1))
    assert pts.shape[0] == corners.shape[0]
    assert np.all(d.min(axis=1) <= 1.0), pts[d.min(axis=1) > 1.0]  # every pick at a corner
    assert np.all(d.min(axis=0) <= 1.0), corners[d.min(axis=0) > 1.0]  # every corner picked
    gftt = cv2.goodFeaturesToTrack(img, 100, 0.01, 3, blockSize=block, useHarrisDetector=False).reshape(-1, 2)
    assert sorted(map(tuple, pts)) == sorted(map(tuple, gftt.astype(np.float64)))


def test_constant_image_gives_nothing():
    for v in (0, 77, 255):
        out = sr.select(np.full((120, 150), v, dtype=np.uint8), sr.Options(cell=16))
        assert out["points"].shape == (0, 2) and out["picks"]["cell"].size == 0


def test_ties_go_to_the_lowest_index():
    # two copies of one square inside one 64-px cell: equal scores, the pick is the smaller y * w + x
    img = _squares((128, 128), [(10, 30, 8), (40, 12, 8)])
    out = sr.select(img, sr.Options(cell=64, block=5))
    p = out["picks"]
    first = p["cell"] == 0
    assert first.sum() == 1
    score = out["score"]
    ys, xs = np.nonzero(sr.candidates(score, 5) & (score == p["score"][first][0]))
    inside = (ys < 64) & (xs < 64)
    assert inside.sum() >= 2  # the tie is real
    assert (p["y"][first][0], p["x"][first][0]) == min(zip(ys[inside], xs[inside]))
    # the max_points cut between equal scores keeps the smaller cell indices
    img = _squares((96, 160), [(8 + 32 * i, 40, 12) for i in range(5)])
    all_ = sr.select(img, sr.Options(cell=32, block=5, quality=1.0))
    assert all_["points"].shape[0] >= 4
    two = sr.select(img, sr.Options(cell=32, block=5, quality=1.0, max_points=2))
    assert np.array_equal(two["points"], all_["points"][:2])


def test_threshold_and_max_points():
    # a bright and a faint square: the faint one's corners score (10 / 255)^2 of the bright one's
    img = _squares((160, 220), [(20, 30, 50)])
    img[70:120, 120:170] = 10
    for q in (0.01, 0.001, 1.0, 0.5):
        out = sr.select(img, sr.Options(cell=16, quality=q))
        ps, kept = out["picks"]["score"], out["kept"]
        thr = np.float32(q) * ps.max()
        assert np.array_equal(kept, ps >= thr), q
    faint = sr.select(img, sr.Options(cell=16, quality=0.001))["points"]
    bright = sr.select(img, sr.Options(cell=16, quality=0.01))["points"]
    assert np.any(faint[:, 0] > 110) and not np.any(bright[:, 0] > 110)
    # max_points: the greatest scores stay, in cell order
    img = _noise((200, 260), 7)
    full = sr.select(img, sr.Options(cell=16, quality=1e-6))
    ps, kept = full["picks"]["score"], full["kept"]
    assert kept.sum() > 40
    cut = sr.select(img, sr.Options(cell=16, quality=1e-6, max_points=40))
    k = np.flatnonzero(kept)
    top = np.sort(k[np.lexsort((full["picks"]["cell"][k], -ps[k]))[:40]])
    assert np.array_equal(np.flatnonzero(cut["kept"]), top)
    assert np.all(np.diff(cut["picks"]["cell"][cut["kept"]]) > 0)


def test_forward_backward_composition():
    clip = rr.Clip(320, 240, 2, delay=0.02, seed=2)
    a, b = clip.render(0), clip.render(1)
    pts = sr.select(a, sr.Options(cell=16))["points"]
    assert pts.shape[0] > 50
    out = sr.forward_backward(a, b, pts, fb_max=1.0)
    fwd = tr.track(a, b, pts)
    assert np.array_equal(out["status"] > 0, fwd["status"])
    back = tr.track(b, a, fwd["tracked"][fwd["status"]])
    k = np.flatnonzero(fwd["status"])
    assert np.array_equal(np.isfinite(out["fb"][k]), back["status"])
    fb = np.hypot(*(back["tracked"][back["status"]] - pts[k[back["status"]]]).T)
    assert np.allclose(out["fb"][k[back["status"]]], fb, rtol=0, atol=1e-12)
    # the rendered motion is smooth: nearly every point returns
    assert np.mean(out["status"][k] == 1) > 0.95
    none = sr.forward_backward(a, b, pts, fb_max=0.0)
    assert np.array_equal(none["status"], fwd["status"].astype(np.uint8)) and np.all(np.isnan(none["fb"]))


def test_symbols_exported_and_declared():
    lib = rsb.load_library()
    name = "rssync_track_frames_ex_device"
    assert name in declared_symbols() and name in rsb.C_ABI_SYMBOLS
    assert hasattr(lib, name)
    header = open(rsb.__file__.replace("rs-sync_b200/__init__.py", "include/rssync_b200.h")).read()
    assert "typedef struct rssync_track_options" in header
    assert [f[0] for f in rsb.TrackOptions._fields_] == ["cell", "block", "quality", "max_points", "fb_max"]
    o = rsb.TrackOptions()
    assert (o.cell, o.block, o.quality, o.max_points, o.fb_max) == (128, 5, 0.01, 512, 1.0)
