"""rssync_track_frames16_device / SyncProblem.track_frames_ex on uint16 planes: byte-for-byte identity with the
8-bit entry point on shifted planes (every output and the problem state); true 10-bit content against the
restatements (tests/select_reference.py, tests/track_reference.py) on the scaled float32 image, and P010 against
the LSB-aligned layout; a low-contrast scene quantised to 10 bits and narrowed to 8 bits against the true
correspondences; a 10-bit clip end to end; the rejections; a multi-device problem."""
import importlib

import numpy as np
import pytest

import render_reference as rr
import select_reference as sr
import track_reference as tr

torch = pytest.importorskip("torch")
from test_gpu_readout_search import _state  # noqa: E402
from test_gpu_track_frames import (BORDER_MARGIN, EIG_MARGIN, STOP_MARGIN, _plane, _problem,  # noqa: E402
                                   _query)

pytestmark = pytest.mark.gpu
rsb = importlib.import_module("rs-sync_b200")
DEV = "cuda:0"


class DeepClip(rr.Clip):
    """rr.Clip rendered at `bits` bits: round((127.5 + contrast * 40 s / norm) * 2^(bits - 8)) clipped to
    [0, 2^bits - 1], s the texture's sum of sinusoids (render_reference.Clip.texture with the contrast scaled
    about mid-grey)"""

    def __init__(self, *a, bits=10, contrast=1.0, **k):
        super().__init__(*a, **k)
        self.bits, self.contrast = bits, contrast

    def render_levels(self, j, device):
        # mirrors render_reference.Clip.render_torch (same chunking and sums) at another depth and contrast
        if not hasattr(self, "_rays_t") or self._rays_t.device != torch.device(device):
            self._rays_t = torch.from_numpy(self._pixel_rays()).to(device)
            self._k_t = torch.from_numpy(self.k).to(device)
            self._ph_t = torch.from_numpy(self.phase).to(device)
            self._amp_t = torch.from_numpy(self.amp).to(device)
        rot = torch.from_numpy(self._row_rotations(j)).to(device)
        out = torch.empty((self.height, self.width), dtype=torch.int32, device=device)
        step = max(1, (1 << 22) // (self.width * 48))
        top = (1 << self.bits) - 1
        for y0 in range(0, self.height, step):
            d = torch.einsum("yij,yxj->yxi", rot[y0:y0 + step], self._rays_t[y0:y0 + step])
            s = (torch.sin(d @ self._k_t.T + self._ph_t) * self._amp_t).sum(-1)
            v = (127.5 + self.contrast * 40.0 * s / self.norm) * 2.0 ** (self.bits - 8)
            out[y0:y0 + step] = torch.clamp(torch.round(v), 0, top).to(torch.int32)
        return out.cpu().numpy().astype(np.uint16)

    def render_host(self):
        """(n_images, height, width) uint16 numpy array of the samples"""
        return np.stack([self.render_levels(j, DEV) for j in range(self.n_images)])


def _u16(host, pad=0):
    """a CUDA uint16 tensor of a (n, h, w) numpy array; pad > 0: rows of w + pad samples (a padded pitch)"""
    if not pad:
        return torch.from_numpy(np.ascontiguousarray(host, dtype=np.uint16)).to(DEV)
    n, h, w = host.shape
    full = np.zeros((n, h, w + pad), dtype=np.uint16)
    full[:, :, :w] = host
    return torch.from_numpy(full).to(DEV)[:, :, :w]


def _ex(p, clip, imgs, shift=None, j0=0, n=None, options=None, params=None, points=None, counts=None):
    n = clip.n_images - 1 - j0 if n is None else n
    r = p.track_frames_ex(clip.frame_ids()[j0:j0 + n], clip.image_ts()[j0:j0 + n + 1], imgs[j0:j0 + n + 1],
                          clip.lens(), params, options, points, counts, shift=shift)
    return dict(points=r.points.cpu().numpy(), counts=r.counts, tracked=r.tracked.cpu().numpy(),
                status=r.status.cpu().numpy(), fb=r.fb_error.cpu().numpy())


def _split(x, counts):
    at = np.concatenate([[0], np.cumsum(counts)])
    return [x[at[i]:at[i + 1]] for i in range(len(counts))]


def _after(p):
    """frame table, arena and device buffers, re-timing table and row fractions"""
    return _state(p), p.retime_table().tobytes(), _plane(p)


def _assert_same(a, b, what):
    for k in a:
        assert a[k].tobytes() == b[k].tobytes(), (what, k)


@pytest.fixture(scope="module")
def clip8():
    c = rr.Clip(1001, 757, 4, delay=0.02, seed=2)
    imgs = c.render_all(DEV)
    return c, imgs, imgs.cpu().numpy()


@pytest.mark.parametrize("shift", [0, 2, 8])
def test_shifted_planes_equal_8bit(clip8, shift):
    """v = P << shift through the 16-bit entry point == P through the 8-bit one: outputs and state"""
    clip, imgs, host = clip8
    wide = _u16(host.astype(np.uint16) << shift)
    n_cases = 0
    for block in (3, 5, 7):
        for cell in (16, 128):
            for fb_max in (0.0, 1.0):
                opt = rsb.TrackOptions(cell=cell, block=block, fb_max=fb_max)
                a, b = _problem(clip), _problem(clip)
                ra, rb = _ex(a, clip, imgs, options=opt), _ex(b, clip, wide, shift, options=opt)
                assert ra["counts"].sum() > 50
                _assert_same(ra, rb, (block, cell, fb_max))
                assert _after(a) == _after(b), (block, cell, fb_max)
                n_cases += 1
    query = _query(clip, clip.n_images - 1, 40)
    counts = np.array([q.shape[0] for q in query])
    pts = torch.from_numpy(np.concatenate(query)).to(DEV)
    for fb_max in (0.0, 1.0):
        opt = rsb.TrackOptions(fb_max=fb_max)
        a, b = _problem(clip), _problem(clip)
        ra = _ex(a, clip, imgs, options=opt, points=pts, counts=counts)
        rb = _ex(b, clip, wide, shift, options=opt, points=pts, counts=counts)
        _assert_same(ra, rb, ("points", fb_max))
        assert _after(a) == _after(b), ("points", fb_max)
        n_cases += 1
    # a padded pitch (rows of width + 37 samples)
    padded = _u16(host.astype(np.uint16) << shift, pad=37)
    assert padded.stride(1) == clip.width + 37
    opt = rsb.TrackOptions(cell=32, block=5, fb_max=1.0)
    a, b = _problem(clip), _problem(clip)
    ra, rb = _ex(a, clip, imgs, options=opt), _ex(b, clip, padded, shift, options=opt)
    _assert_same(ra, rb, "padded")
    assert _after(a) == _after(b)
    print(f"shift {shift}: {n_cases + 1} configurations identical to the 8-bit path")


def test_shifted_planes_across_chunks():
    """41 images at 2.7k take two pyramid chunks"""
    clip = rr.Clip(2704, 2028, 41, delay=0.02, seed=4)
    imgs = clip.render_all(DEV)
    wide = _u16(imgs.cpu().numpy().astype(np.uint16) << 8)
    opt = rsb.TrackOptions(cell=64, block=5, fb_max=1.0)
    a, b = _problem(clip), _problem(clip)
    ra, rb = _ex(a, clip, imgs, options=opt), _ex(b, clip, wide, 8, options=opt)
    assert ra["counts"].sum() > 1000
    _assert_same(ra, rb, "chunks")
    assert _after(a) == _after(b)


@pytest.fixture(scope="module")
def clip10():
    c = DeepClip(1001, 757, 3, delay=0.02, seed=2, bits=10)
    return c, c.render_host()


def test_p010_equals_lsb(clip10):
    clip, x = clip10
    assert np.unique(x).size > 256  # more levels than 8 bits hold
    lsb, p010 = _u16(x), _u16(x << 6)
    for opt in (rsb.TrackOptions(cell=32, fb_max=1.0), rsb.TrackOptions(cell=128, block=7, fb_max=0.0)):
        a, b = _problem(clip), _problem(clip)
        ra, rb = _ex(a, clip, lsb, 2, options=opt), _ex(b, clip, p010, 8, options=opt)
        _assert_same(ra, rb, "p010")
        assert _after(a) == _after(b)


def test_10bit_selection_matches_restatement(clip10):
    clip, x = clip10
    imgs = _u16(x)
    f = x.astype(np.float32) * np.float32(0.25)
    p = _problem(clip)
    for block in (3, 5, 7):
        score = [sr.scores(h, block) for h in f[:-1]]
        for cell in (16, 128):
            got = _ex(p, clip, imgs, 2, options=rsb.TrackOptions(cell=cell, block=block, fb_max=0.0))
            for j, pts in enumerate(_split(got["points"], got["counts"])):
                ref = sr.select(f[j], sr.Options(cell=cell, block=block), score[j])["points"]
                assert pts.tobytes() == ref.tobytes(), (block, cell, j, pts.shape, ref.shape)


def test_10bit_positions_match_restatement(clip10):
    """the tolerances and stop-margin handling of test_gpu_track_frames.test_positions_match_restatement"""
    clip, x = clip10
    imgs = _u16(x)
    f = x.astype(np.float32) * np.float32(0.25)
    query = _query(clip, clip.n_images - 1, max(20, clip.width // 14))
    counts = np.array([q.shape[0] for q in query])
    got = _ex(_problem(clip), clip, imgs, 2, options=rsb.TrackOptions(fb_max=0.0),
              points=torch.from_numpy(np.concatenate(query)).to(DEV), counts=counts)
    n_near = n_stop_near = n_both = 0
    for j, (q, t, s) in enumerate(zip(query, *[_split(got[k], counts) for k in ("tracked", "status")])):
        ref = tr.track(f[j], f[j + 1], q)
        s = s.astype(bool)
        both = s & ref["status"]
        assert both.sum() >= 0.9 * q.shape[0] - 8
        err = np.hypot(*(t[both] - ref["tracked"][both]).T)
        stop_near = ref["stop_margin"][both] < STOP_MARGIN
        assert err[~stop_near].max() <= 1e-3, (j, err[~stop_near].max())
        assert np.all(err[stop_near] <= 0.1), (j, err[stop_near].max())
        n_stop_near += int(np.sum(err[stop_near] > 1e-3))
        n_both += int(both.sum())
        differ = s != ref["status"]
        near = (ref["eig_margin"] < EIG_MARGIN) | (np.abs(np.nan_to_num(ref["border_margin"], nan=1.0)) < BORDER_MARGIN)
        assert not np.any(differ & ~near), np.flatnonzero(differ & ~near)
        n_near += int(differ.sum())
    print(f"10-bit: {n_both} points kept by both, {n_stop_near} beyond 1e-3 px next to the epsilon stop, "
          f"{n_near} status differences next to a threshold")
    assert n_near <= 2 and n_stop_near <= max(2, n_both // 50)


def _errors(clip, res):
    errs = []
    for j, (q, t, s) in enumerate(zip(*[_split(res[k], res["counts"]) for k in ("points", "tracked", "status")])):
        k = s == 1
        errs.append(np.hypot(*(t[k] - clip.true_b(j, q[k])).T))
    e = np.concatenate(errs)
    return float(np.median(e)), float(np.percentile(e, 90)), int(e.size)


def test_low_contrast_10bit_against_8bit():
    """the texture at 1/8 of its contrast about mid-grey, quantised to 10 bits, and the same samples narrowed
    to 8 bits (x >> 2, what a caller of the 8-bit entry point does): errors against the true correspondences
    and kept points, on the 200-px grid and with the selection, the backward check on"""
    clip = DeepClip(2704, 2028, 9, delay=0.02, seed=5, bits=10, contrast=0.125)
    x = clip.render_host()
    assert 300 < x.min() and x.max() < 730  # an 8-bit amplitude of 5 grey levels times the texture's peaks
    ten, eight = _u16(x), torch.from_numpy((x >> 2).astype(np.uint8)).to(DEV)
    grid = rsb.grid_points(clip.width, clip.height, 200)
    n = clip.n_images - 1
    counts = np.full(n, grid.shape[0])
    pts = torch.from_numpy(np.concatenate([grid] * n)).to(DEV)
    opt_sel = rsb.TrackOptions(cell=128, max_points=grid.shape[0], fb_max=1.0)
    out = {}
    for name, kw in (("grid", dict(options=rsb.TrackOptions(fb_max=1.0), points=pts, counts=counts)),
                     ("selection", dict(options=opt_sel))):
        r10 = _errors(clip, _ex(_problem(clip), clip, ten, 2, **kw))
        r8 = _errors(clip, _ex(_problem(clip), clip, eight, **kw))
        out[name] = (r10, r8)
        print(f"low contrast, {name}: 10-bit median {r10[0]:.4f} px, p90 {r10[1]:.4f} px, kept {r10[2]}; "
              f"8-bit median {r8[0]:.4f} px, p90 {r8[1]:.4f} px, kept {r8[2]}")
    for name, (r10, r8) in out.items():
        assert r10[0] <= r8[0] and r10[1] <= r8[1] and r10[2] >= r8[2], (name, r10, r8)


def test_10bit_end_to_end():
    """a 10-bit 2.7k clip, 121 images, true delay 37 ms: selection and the backward check, then PreSync and
    4 x Sync"""
    clip = DeepClip(2704, 2028, 121, delay=0.037, seed=5, bits=10)
    imgs = _u16(clip.render_host())
    budget = rsb.grid_points(clip.width, clip.height, 200).shape[0]
    opt = rsb.TrackOptions(cell=128, max_points=budget, fb_max=1.0)
    p = _problem(clip)
    for j0 in range(0, 120, 64):
        _ex(p, clip, imgs, 2, j0, min(64, 120 - j0), options=opt)
    fb, fe = int(clip.frame_ids()[0]), int(clip.frame_ids()[-1]) + 1
    step, radius = 0.002, 0.2
    c, d = p.PreSync(0.0, fb, fe, step, radius)
    assert abs(d - clip.delay) <= step + 1e-12, d
    for _ in range(4):
        c, d = p.Sync(d, fb, fe, 0.0, radius)
    print(f"10-bit end to end: PreSync then 4 x Sync delay {d * 1e3:.4f} ms (true {clip.delay * 1e3:.1f} ms)")
    assert abs(d - clip.delay) < 0.5e-3, d


def _assert_rejected(p, code, text, fn):
    before = (p.frame_table().tobytes(), p.call_counter(), p.retime_table().tobytes(), _state(p))
    with pytest.raises(rsb.RsSyncError) as e:
        fn()
    assert e.value.code == code and text in e.value.message, (e.value.code, e.value.message)
    assert (p.frame_table().tobytes(), p.call_counter(), p.retime_table().tobytes(), _state(p)) == before


def test_errors_apply_nothing():
    clip = rr.Clip(320, 240, 4, delay=0.02, seed=2)
    imgs = _u16(clip.render_all(DEV).cpu().numpy().astype(np.uint16) << 8)
    p = _problem(clip)
    _ex(p, clip, imgs, 8, 0, 1, options=rsb.TrackOptions(cell=32))  # something to leave unchanged
    fr, ts, lens = clip.frame_ids()[:2], clip.image_ts()[:3], clip.lens()
    L = rsb.load_library()
    out = torch.empty((2 * 512, 2), dtype=torch.float64, device=DEV)
    host_img = imgs.cpu().numpy()

    def call(shift=8, options=rsb.TrackOptions(), points=None, counts=None, width=None, height=None, pitch=None,
             params=None, ts=ts, lens=lens, image_ptr=None):
        cn = None if counts is None else np.ascontiguousarray(counts, dtype=np.uint64)
        t = np.ascontiguousarray(ts, dtype=np.float64)
        rc = L.rssync_track_frames16_device(
            p.h, 2, np.ascontiguousarray(fr).ctypes.data_as(rsb.c_i64_p),
            None if cn is None else cn.ctypes.data_as(rsb.C.POINTER(rsb.C.c_size_t)), t.ctypes.data_as(rsb.c_double_p),
            None if points is None else rsb.C.c_void_p(points.data_ptr() if hasattr(points, "data_ptr")
                                                       else points.ctypes.data),
            rsb.C.c_void_p(imgs.data_ptr() if image_ptr is None else image_ptr),
            2 * imgs.stride(1) if pitch is None else pitch, clip.width if width is None else width,
            clip.height if height is None else height, shift, rsb.C.byref(rsb.Lens(*lens)),
            None if params is None else rsb.C.byref(params), rsb.C.byref(options), rsb.C.c_void_p(out.data_ptr()),
            None, None, None, None, None)
        p._check(rc)

    # the 16-bit checks
    for s in (-1, 9, 16):
        _assert_rejected(p, rsb.E_INVALID, "shift outside 0..8", lambda: call(shift=s))
    _assert_rejected(p, rsb.E_INVALID, "2-byte aligned", lambda: call(image_ptr=imgs.data_ptr() + 1))
    _assert_rejected(p, rsb.E_INVALID, "even pitch", lambda: call(pitch=2 * clip.width + 1))
    _assert_rejected(p, rsb.E_INVALID, "even pitch", lambda: call(pitch=2 * clip.width - 2))
    # the ex form's checks, reached through the 16-bit entry point
    _assert_rejected(p, rsb.E_INVALID, "pitch below width", lambda: call(pitch=clip.width - 2))
    _assert_rejected(p, rsb.E_INVALID, "images is not device memory", lambda: call(image_ptr=host_img.ctypes.data))
    for bad in (dict(cell=15), dict(block=4), dict(quality=0.0), dict(max_points=513), dict(fb_max=-1.0)):
        _assert_rejected(p, rsb.E_INVALID, "options out of range", lambda: call(options=rsb.TrackOptions(**bad)))
    pts = torch.zeros((4, 2), dtype=torch.float64, device=DEV)
    _assert_rejected(p, rsb.E_INVALID, "both be given or both be NULL", lambda: call(points=pts))
    _assert_rejected(p, rsb.E_INVALID, "both be given or both be NULL", lambda: call(counts=[2, 2]))
    _assert_rejected(p, rsb.E_INVALID, "points is not device memory",
                     lambda: call(points=np.zeros((4, 2)), counts=[2, 2]))
    _assert_rejected(p, rsb.E_INVALID, "more than 512", lambda: call(points=pts, counts=[513, 1]))
    _assert_rejected(p, rsb.E_INVALID, "parameters out of range", lambda: call(params=rsb.TrackParams(levels=0)))
    _assert_rejected(p, rsb.E_INVALID, "image smaller", lambda: call(width=83, pitch=2 * clip.width))
    small = rsb.TrackParams(levels=1, window=5)
    _assert_rejected(p, rsb.E_INVALID, "2 * (block / 2 + 2) + 1",
                     lambda: call(width=8, params=small, options=rsb.TrackOptions(block=5)))
    _assert_rejected(p, rsb.E_INVALID, "bad lens profile", lambda: call(lens=(0.011, 0.0) + tuple(lens[2:])))
    t = ts.copy()
    t[0] = np.nan
    _assert_rejected(p, rsb.E_NONFINITE, "ts_a", lambda: call(ts=t))
    nan_pts = torch.zeros((4, 2), dtype=torch.float64, device=DEV) + 50.0
    nan_pts[1, 0] = float("nan")
    _assert_rejected(p, rsb.E_NONFINITE, "non-finite numbers in rays_a", lambda: call(points=nan_pts, counts=[2, 2]))
    # the Python front: uint16 needs a shift, uint8 takes none
    with pytest.raises(ValueError, match="need a shift"):
        _ex(p, clip, imgs, None, 0, 1)
    with pytest.raises(ValueError, match="uint16 images only"):
        _ex(p, clip, clip.render_all(DEV), 2, 0, 1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_multi_device_equals_single(clip10):
    clip, x = clip10
    imgs = _u16(x)
    one, multi = _problem(clip), _problem(clip, devices=[0, 1])
    opt = rsb.TrackOptions(cell=64, fb_max=1.0)
    a, b = _ex(one, clip, imgs, 2, options=opt), _ex(multi, clip, imgs, 2, options=opt)
    _assert_same(a, b, "multi")
    fb, fe = int(clip.frame_ids()[0]), int(clip.frame_ids()[-1]) + 1
    for p in (one, multi):
        p.set_rng(100, 3)
    assert one.PreSync(0.0, fb, fe, 0.002, 0.1) == multi.PreSync(0.0, fb, fe, 0.002, 0.1)
    r = [0.0, 0.008, 0.011, 0.014]
    x1, y1 = one.readout_search(r, 0.0, fb, fe, 0.002, 0.1), multi.readout_search(r, 0.0, fb, fe, 0.002, 0.1)
    assert all(np.array_equal(u, v) for u, v in zip(x1, y1))
