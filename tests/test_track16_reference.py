"""The exactness the 16-bit tracking entry point (rssync_track_frames16_device) rests on, on the CPU: a 16-bit
plane v = P << shift read as (float)v * 2^-shift gives the 8-bit plane P's float32 intensities, so the tracker
and selection restatements (tests/track_reference.py, tests/select_reference.py) give identical bits on both;
likewise a P010 plane (x << 6, shift 8) and the LSB-aligned plane x (shift 2).  And the new C symbol."""
import importlib

import numpy as np
import pytest

import render_reference as rr
import select_reference as sr
import track_reference as tr
from test_abi import declared_symbols

rsb = importlib.import_module("rs-sync_b200")


def level0(v, shift):
    """the contract's level-0 intensity of a 16-bit plane: (float)v * 2^-shift in float32"""
    return np.asarray(v).astype(np.float32) * np.float32(2.0 ** -shift)


@pytest.fixture(scope="module")
def frames():
    clip = rr.Clip(320, 240, 2, delay=0.02, seed=2)
    return clip.render(0), clip.render(1)


@pytest.mark.parametrize("shift", [0, 2, 4, 8])
def test_shifted_planes_give_identical_bits(frames, shift):
    a, b = frames
    va, vb = (x.astype(np.uint16) << shift for x in (a, b))
    fa, fb = level0(va, shift), level0(vb, shift)
    assert fa.tobytes() == a.astype(np.float32).tobytes() and fb.tobytes() == b.astype(np.float32).tobytes()
    for block in (3, 5, 7):
        s8, s16 = sr.scores(a, block), sr.scores(fa, block)
        assert s8.tobytes() == s16.tobytes(), block
        opt = sr.Options(cell=16, block=block)
        assert sr.select(a, opt, s8)["points"].tobytes() == sr.select(fa, opt, s16)["points"].tobytes(), block
    pts = sr.select(a, sr.Options(cell=16))["points"]
    assert pts.shape[0] > 50
    r8, r16 = sr.forward_backward(a, b, pts, fb_max=1.0), sr.forward_backward(fa, fb, pts, fb_max=1.0)
    assert r8["status"].tobytes() == r16["status"].tobytes()
    assert r8["fb"].tobytes() == r16["fb"].tobytes()
    assert r8["forward"]["tracked"].tobytes() == r16["forward"]["tracked"].tobytes()


def test_p010_equals_lsb_aligned():
    """10-bit samples over the whole range: x << 6 at shift 8 and x at shift 2 give the same intensities, and
    every 16-bit sample times 2^-shift is exact for every shift"""
    x = np.arange(1024, dtype=np.uint16)
    assert level0(x << 6, 8).tobytes() == level0(x, 2).tobytes()
    assert np.array_equal(level0(x, 2).astype(np.float64), x / 4.0)
    v = np.arange(65536, dtype=np.uint32)
    for shift in range(9):
        assert np.array_equal(level0(v, shift).astype(np.float64), v / 2.0 ** shift), shift


def test_symbol_exported_and_declared():
    name = "rssync_track_frames16_device"
    assert name in declared_symbols() and name in rsb.C_ABI_SYMBOLS
    assert hasattr(rsb.load_library(), name)
