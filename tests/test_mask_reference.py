"""The mask restatement (tests/mask_reference.py) on the CPU: eligibility equals cv2.erode, the masked selection
with nothing masked equals select_reference's, a cell whose only candidates are masked has no pick, the quality
threshold sees only eligible picks; and the new C symbol."""
import importlib

import numpy as np
import pytest

import mask_reference as mr
import render_reference as rr
import select_reference as sr
from test_abi import declared_symbols

cv2 = pytest.importorskip("cv2")
rsb = importlib.import_module("rs-sync_b200")


def _masks():
    """random blobs, and zeros on every border, a corner and a single pixel"""
    rng = np.random.default_rng(11)
    h, w = 151, 203
    blobs = np.ones((h, w), dtype=np.uint8)
    for _ in range(12):
        x, y = rng.integers(0, w), rng.integers(0, h)
        blobs[max(0, y - rng.integers(0, 9)):y + rng.integers(1, 9), max(0, x - rng.integers(0, 9)):x + rng.integers(1, 9)] = 0
    borders = np.full((h, w), 7, dtype=np.uint8)
    borders[0, 40:45] = 0
    borders[h - 1, 100] = 0
    borders[60:64, 0] = 0
    borders[90, w - 1] = 0
    corner = np.ones((h, w), dtype=np.uint8)
    corner[h - 3:, w - 2:] = 0
    dot = np.ones((h, w), dtype=np.uint8)
    dot[75, 101] = 0
    return [blobs, borders, corner, dot, rng.integers(0, 2, (h, w), dtype=np.uint8) * 255]


@pytest.mark.parametrize("margin", [0, 1, 11, 63])
def test_eligibility_equals_cv2_erode(margin):
    for m in _masks():
        ref = cv2.erode((m != 0).astype(np.uint8), np.ones((2 * margin + 1, 2 * margin + 1), np.uint8)) != 0
        assert np.array_equal(mr.eligible(m, margin), ref), margin


def test_nearest_pixel():
    q = mr.nearest(np.array([[0.49, 0.5], [2.5, 3.4999], [-0.5, 7.0]]))
    assert q.tolist() == [[0, 1], [3, 3], [0, 7]]


@pytest.fixture(scope="module")
def image():
    return rr.Clip(320, 240, 1, delay=0.02, seed=2).render(0)


@pytest.mark.parametrize("cell,block", [(16, 3), (32, 5), (128, 7)])
def test_all_ones_mask_equals_unmasked_selection(image, cell, block):
    opt = sr.Options(cell=cell, block=block)
    score = sr.scores(image, block)
    ref = sr.select(image, opt, score)["points"]
    got = mr.select(image, mr.eligible(np.ones(image.shape, np.uint8), 40), opt, score)
    assert ref.shape[0] >= 6 and got.tobytes() == ref.tobytes()


def test_masked_cell_has_no_pick(image):
    opt = sr.Options(cell=32, block=5)
    score = sr.scores(image, 5)
    picks = sr.select(image, opt, score)["picks"]
    c = int(picks["cell"][5])
    ncx = (image.shape[1] + 31) // 32
    cy, cx = divmod(c, ncx)
    mask = np.ones(image.shape, np.uint8)
    mask[cy * 32:cy * 32 + 32, cx * 32:cx * 32 + 32] = 0  # every candidate of the cell, nothing else
    got = mr.select(image, mr.eligible(mask, 0), opt, score)
    cells = (got[:, 1].astype(int) // 32) * ncx + got[:, 0].astype(int) // 32
    assert c not in cells
    ref = sr.select(image, opt, score)["points"]
    assert got.shape[0] == ref.shape[0] - 1


def test_threshold_uses_eligible_maximum(image):
    """with quality 0.5, masking the strongest picks lets weaker ones pass: the threshold follows the greatest
    eligible pick"""
    opt = sr.Options(cell=32, block=5, quality=0.5)
    score = sr.scores(image, 5)
    picks = sr.select(image, opt, score)["picks"]
    order = np.argsort(-picks["score"])
    mask = np.ones(image.shape, np.uint8)
    for i in order[:len(order) // 2]:  # the stronger half of the picks masked at the pixel
        mask[picks["y"][i], picks["x"][i]] = 0
    elig = mr.eligible(mask, 0)
    got = mr.select(image, elig, opt, score)
    cand = sr.candidates(score, 5) & elig
    m = score[cand].max()
    s = score[got[:, 1].astype(int), got[:, 0].astype(int)]
    assert np.all(s >= np.float32(0.5) * m)
    assert m < picks["score"].max()
    unmasked = sr.select(image, opt, score)["points"]
    weak = {(x, y) for x, y in got.tolist()} - {(x, y) for x, y in unmasked.tolist()}
    assert weak, "a pick below half the unmasked maximum should pass once the strong picks are masked"


def test_status_rule():
    elig_a = np.ones((10, 12), bool)
    elig_b = np.ones((10, 12), bool)
    elig_a[2, 3] = False
    elig_b[5, 6] = False
    q = np.array([[3.2, 1.6], [1.0, 1.0], [3.0, 2.0], [1.0, 1.0]])
    t = np.array([[1.0, 1.0], [5.6, 5.4], [3.0, 2.0], [1.0, 1.0]])
    st = mr.masked_status(np.array([1, 1, 0, 2]), q, t, elig_a, elig_b)
    assert st.tolist() == [3, 3, 0, 2]


def test_symbol_exported_and_declared():
    name = "rssync_track_frames_masked_device"
    assert name in declared_symbols() and name in rsb.C_ABI_SYMBOLS
    assert hasattr(rsb.load_library(), name)
