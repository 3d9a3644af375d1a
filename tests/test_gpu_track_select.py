"""rssync_track_frames_ex_device / SyncProblem.track_frames_ex on rendered rolling-shutter frames: the device's
point selection against the float32 restatement (tests/select_reference.py), bit for bit; equivalence with
track_frames; the backward pass against the restatement; the ingest of the kept pairs; an occluding block; a
low-texture scene end to end; the rejections; a multi-device problem."""
import importlib

import numpy as np
import pytest

import render_reference as rr
import select_reference as sr

torch = pytest.importorskip("torch")
from test_gpu_readout_search import _state  # noqa: E402
from test_gpu_track_frames import (BORDER_MARGIN, EIG_MARGIN, STOP_MARGIN, _everything, _problem,  # noqa: E402
                                   _query, _run)

pytestmark = pytest.mark.gpu
rsb = importlib.import_module("rs-sync_b200")
DEV = "cuda:0"


def _ex(p, clip, imgs, j0=0, n=None, options=None, params=None, points=None, counts=None):
    n = clip.n_images - 1 - j0 if n is None else n
    r = p.track_frames_ex(clip.frame_ids()[j0:j0 + n], clip.image_ts()[j0:j0 + n + 1], imgs[j0:j0 + n + 1],
                          clip.lens(), params, options, points, counts)
    return dict(points=r.points.cpu().numpy(), counts=r.counts, tracked=r.tracked.cpu().numpy(),
                status=r.status.cpu().numpy(), fb=r.fb_error.cpu().numpy())


def _split(x, counts):
    at = np.concatenate([[0], np.cumsum(counts)])
    return [x[at[i]:at[i + 1]] for i in range(len(counts))]


@pytest.fixture(scope="module")
def clips():
    out = {}
    for W, H, n in ((320, 240, 3), (2704, 2028, 3), (1001, 757, 3)):
        c = rr.Clip(W, H, n, delay=0.02, seed=2)
        out[(W, H)] = (c, c.render_all(DEV))
    return out


@pytest.mark.parametrize("size", [(320, 240), (2704, 2028), (1001, 757)])
def test_selection_matches_restatement(clips, size):
    clip, imgs = clips[size]
    host = imgs.cpu().numpy()
    p = _problem(clip)
    for block in (3, 5, 7):
        score = [sr.scores(h, block) for h in host[:-1]]
        for cell in (16, 64, 128):
            for mp in ((512, 37) if cell == 16 else (512,)):  # (37: the max_points cut)
                opt = rsb.TrackOptions(cell=cell, block=block, max_points=mp, fb_max=0.0)
                got = _ex(p, clip, imgs, options=opt)
                for j, pts in enumerate(_split(got["points"], got["counts"])):
                    ref = sr.select(host[j], sr.Options(cell=cell, block=block, max_points=mp), score[j])["points"]
                    assert pts.tobytes() == ref.tobytes(), (size, block, cell, mp, j, pts.shape, ref.shape)
    print(f"{size}: selection identical to the restatement for blocks 3, 5, 7, cells 16, 64, 128")


def test_selection_across_chunks():
    """41 images at 2.7k take two pyramid chunks; batches of 6 frames take one each"""
    clip = rr.Clip(2704, 2028, 41, delay=0.02, seed=4)
    imgs = clip.render_all(DEV)
    opt = rsb.TrackOptions(cell=64, block=5, fb_max=1.0)
    one = _ex(_problem(clip), clip, imgs, options=opt)
    many = _problem(clip)
    parts = [_ex(many, clip, imgs, j0, min(6, 40 - j0), options=opt) for j0 in range(0, 40, 6)]
    for k in ("points", "tracked", "status", "fb", "counts"):
        assert np.concatenate([x[k] for x in parts]).tobytes() == one[k].tobytes(), k
    host = imgs.cpu().numpy()
    pts = _split(one["points"], one["counts"])
    for j in (0, 37, 38, 39):
        ref = sr.select(host[j], sr.Options(cell=64, block=5))["points"]
        assert pts[j].tobytes() == ref.tobytes(), j


@pytest.fixture(scope="module")
def clip30():
    c = rr.Clip(676, 507, 31, delay=0.031, seed=3)
    return c, c.render_all(DEV)


def test_caller_points_without_backward_equal_track_frames(clip30):
    clip, imgs = clip30
    query = _query(clip, 30, 50)
    counts = np.array([q.shape[0] for q in query])
    pts = torch.from_numpy(np.concatenate(query)).to(DEV)
    a, b = _problem(clip), _problem(clip)
    tracked, status, _ = _run(a, clip, imgs, query)
    got = _ex(b, clip, imgs, options=rsb.TrackOptions(fb_max=0.0), points=pts, counts=counts)
    assert got["tracked"].tobytes() == tracked.tobytes()
    assert np.array_equal(got["status"], status.astype(np.uint8))
    assert np.array_equal(got["points"], np.concatenate(query)) and np.array_equal(got["counts"], counts)
    assert np.all(np.isnan(got["fb"]))
    fb, fe = int(clip.frame_ids()[0]), int(clip.frame_ids()[-1]) + 1
    ra, rb = _everything(a, fb, fe), _everything(b, fb, fe)
    assert [k for k in ra if ra[k] != rb[k]] == []


@pytest.mark.parametrize("size", [(320, 240), (2704, 2028)])
def test_backward_matches_restatement(clips, size):
    clip, imgs = clips[size]
    host = imgs.cpu().numpy()
    fb_max = 0.05  # small enough that the rendered scene rejects some points
    got = _ex(_problem(clip), clip, imgs, options=rsb.TrackOptions(cell=32, fb_max=fb_max))
    n_fb = n_far = n_status = n_near = 0
    for j, (q, t, s, f) in enumerate(zip(*[_split(got[k], got["counts"]) for k in ("points", "tracked", "status",
                                                                                    "fb")])):
        ref = sr.forward_backward(host[j], host[j + 1], q, fb_max=fb_max)
        fwd = ref["forward"]
        fnear = (fwd["eig_margin"] < EIG_MARGIN) | (np.abs(np.nan_to_num(fwd["border_margin"], nan=1.0)) < BORDER_MARGIN)
        fstop = fwd["stop_margin"] < STOP_MARGIN
        both = np.isfinite(f) & np.isfinite(ref["fb"])
        bstop = np.zeros(q.shape[0], dtype=bool)
        bnear = np.zeros(q.shape[0], dtype=bool)
        if ref["backward"] is not None:
            k = np.flatnonzero(fwd["status"])
            bstop[k] = ref["backward"]["stop_margin"] < STOP_MARGIN
            bnear[k] = (ref["backward"]["eig_margin"] < EIG_MARGIN) | (
                np.abs(np.nan_to_num(ref["backward"]["border_margin"], nan=1.0)) < BORDER_MARGIN)
        err = np.abs(f[both] - ref["fb"][both])
        near_stop = (fstop | bstop)[both]
        assert np.all(err[~near_stop] <= 1e-3), err[~near_stop].max()
        assert np.all(err[near_stop] <= 0.2), err[near_stop].max()
        n_far += int(np.sum(err[near_stop] > 1e-3))
        n_fb += int(both.sum())
        # status 2 agrees, except next to fb_max or next to a threshold of either pass
        edge = (np.abs(np.nan_to_num(ref["fb"], nan=10.0) - fb_max) <= 1e-3) | fnear | bnear | fstop | bstop
        differ = s != ref["status"]
        assert not np.any(differ & ~edge), np.flatnonzero(differ & ~edge)
        n_near += int(differ.sum())
        n_status += int(np.sum(s == 2))
    print(f"{size}: {n_fb} backward distances, {n_far} beyond 1e-3 px next to the epsilon stop; {n_status} "
          f"rejected; {n_near} status differences next to a threshold")
    assert n_fb > 100 and n_far <= max(2, n_fb // 50) and n_near <= max(2, n_fb // 100)


def test_ingest_identity_with_selection_and_backward(clip30):
    clip, imgs = clip30
    a = _problem(clip)
    got = _ex(a, clip, imgs, options=rsb.TrackOptions(cell=32, fb_max=0.05))
    assert np.any(got["status"] == 2) and np.any(got["status"] == 1)
    keep = got["status"] == 1
    kept = np.array([int(s.sum()) for s in _split(keep, got["counts"])])
    b = _problem(clip)
    ts = clip.image_ts()
    b.set_track_pixels(clip.frame_ids(), kept, ts[:-1], ts[1:], torch.from_numpy(got["points"][keep]).to(DEV),
                       torch.from_numpy(got["tracked"][keep]).to(DEV), clip.lens(), clip.height)
    assert list(a.frame_table()["n"]) == list(kept)
    fb, fe = int(clip.frame_ids()[0]), int(clip.frame_ids()[-1]) + 1
    ra, rb = _everything(a, fb, fe), _everything(b, fb, fe)
    assert [k for k in ra if ra[k] != rb[k]] == []


def test_occluding_block():
    """a seeded 400 x 400 noise block pasted into image i + 1 at 2.7k: the backward check rejects the points
    whose true position falls in it and keeps the points a window or more away"""
    clip = rr.Clip(2704, 2028, 4, delay=0.02, seed=6)
    imgs = clip.render_all(DEV)
    rng = np.random.default_rng(77)
    blocks = [(900, 700), (1500, 1100), (1200, 500)]
    occl = imgs.clone()
    for j, (bx, by) in enumerate(blocks):
        occl[j + 1, by:by + 400, bx:bx + 400] = torch.from_numpy(rng.integers(0, 256, (400, 400), dtype=np.uint8)).to(DEV)
    query, inside, away = [], [], []
    for j, (bx, by) in enumerate(blocks):
        g = rsb.grid_points(700, 700, 32)[:512] + np.array([bx - 150.0, by - 150.0])
        t = clip.true_b(j, g)
        query.append(g)
        inside.append((t[:, 0] >= bx) & (t[:, 0] <= bx + 399) & (t[:, 1] >= by) & (t[:, 1] <= by + 399))
        dx = np.maximum(np.maximum(bx - t[:, 0], t[:, 0] - (bx + 399)), 0)
        dy = np.maximum(np.maximum(by - t[:, 1], t[:, 1] - (by + 399)), 0)
        away.append(np.hypot(dx, dy) >= 21)
    counts = np.array([q.shape[0] for q in query])
    pts = torch.from_numpy(np.concatenate(query)).to(DEV)
    inside, away = np.concatenate(inside), np.concatenate(away)
    fwd = _ex(_problem(clip), clip, occl, options=rsb.TrackOptions(fb_max=0.0), points=pts, counts=counts)
    chk = _ex(_problem(clip), clip, occl, options=rsb.TrackOptions(fb_max=1.0), points=pts, counts=counts)
    kept_fwd = np.mean(fwd["status"][inside] == 1)
    rejected = np.mean(chk["status"][inside] != 1)
    away_kept = np.mean(chk["status"][away] == 1)
    print(f"occlusion: {inside.sum()} points in the block; forward only keeps {kept_fwd:.3f}, the backward check "
          f"rejects {rejected:.3f}; {away.sum()} points a window or more away keep status 1 in {away_kept:.4f}")
    assert inside.sum() > 300 and away.sum() > 300
    assert rejected >= 0.9 and away_kept >= 0.99


class FadingClip(rr.Clip):
    """rr.Clip whose texture contrast fades to flat grey over about half the sphere: full contrast where the
    world direction d has d . axis >= 0.25, none where d . axis <= -0.25, linear between; axis points from the
    first image's centre ray towards its right edge, so the left part of the view is flat"""

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        c = self.world(0, np.array([self.width / 2.0]), np.array([self.height / 2.0]))[0]
        e = self.world(0, np.array([self.width - 1.0]), np.array([self.height / 2.0]))[0]
        ax = e - np.dot(e, c) * c
        self.axis = ax / np.linalg.norm(ax)

    def fade(self, d):
        return np.clip(0.5 + 2.0 * (d @ self.axis), 0.0, 1.0)

    def texture(self, d):
        return 127.5 + (super().texture(d) - 127.5) * self.fade(d)

    def render_torch(self, j, device):
        # mirrors render_reference.Clip.render_torch (same chunking, 40.0 contrast and rounding) with the fade
        # applied to the contrast term; keep the two in step if the base renderer changes
        if not hasattr(self, "_rays_t") or self._rays_t.device != torch.device(device):
            self._rays_t = torch.from_numpy(self._pixel_rays()).to(device)
            self._k_t = torch.from_numpy(self.k).to(device)
            self._ph_t = torch.from_numpy(self.phase).to(device)
            self._amp_t = torch.from_numpy(self.amp).to(device)
            self._ax_t = torch.from_numpy(self.axis).to(device)
        rot = torch.from_numpy(self._row_rotations(j)).to(device)
        out = torch.empty((self.height, self.width), dtype=torch.uint8, device=device)
        step = max(1, (1 << 22) // (self.width * 48))
        for y0 in range(0, self.height, step):
            d = torch.einsum("yij,yxj->yxi", rot[y0:y0 + step], self._rays_t[y0:y0 + step])
            s = (torch.sin(d @ self._k_t.T + self._ph_t) * self._amp_t).sum(-1)
            f = torch.clamp(0.5 + 2.0 * (d @ self._ax_t), 0.0, 1.0)
            out[y0:y0 + step] = torch.clamp(torch.round(127.5 + 40.0 * s / self.norm * f), 0, 255).to(torch.uint8)
        return out


def test_low_texture_scene_end_to_end():
    clip = FadingClip(2704, 2028, 121, delay=0.037, seed=5)
    imgs = clip.render_all(DEV)
    grid = rsb.grid_points(clip.width, clip.height, 200)
    budget = grid.shape[0]
    opt = rsb.TrackOptions(cell=128, max_points=budget, fb_max=1.0)
    # accuracy on the first frames: kept points and the median error against the truth, equal budgets
    eg, es = [], []
    pg, ps = _problem(clip), _problem(clip)
    counts = np.full(8, budget)
    g = _ex(pg, clip, imgs, 0, 8, options=rsb.TrackOptions(fb_max=0.0),
            points=torch.from_numpy(np.concatenate([grid] * 8)).to(DEV), counts=counts)
    s = _ex(ps, clip, imgs, 0, 8, options=opt)
    for j in range(8):
        for res, errs in ((g, eg), (s, es)):
            q, t, st = (_split(res[k], res["counts"])[j] for k in ("points", "tracked", "status"))
            k = st == 1
            errs.append(np.hypot(*(t[k] - clip.true_b(j, q[k])).T))
    ng, ns = sum(e.size for e in eg), sum(e.size for e in es)
    mg, ms = float(np.median(np.concatenate(eg))), float(np.median(np.concatenate(es)))
    print(f"low texture, budget {budget}: grid keeps {ng} points, median error {mg:.4f} px; selection keeps {ns}, "
          f"median error {ms:.4f} px")
    assert ns >= ng and ms <= mg
    # the whole clip with selection and the backward check, then PreSync, 4 x Sync and the readout search
    p = _problem(clip)
    for j0 in range(0, 120, 64):
        _ex(p, clip, imgs, j0, min(64, 120 - j0), options=opt)
    fb, fe = int(clip.frame_ids()[0]), int(clip.frame_ids()[-1]) + 1
    step, radius = 0.002, 0.2
    c, d = p.PreSync(0.0, fb, fe, step, radius)
    assert abs(d - clip.delay) <= step + 1e-12, d
    for _ in range(4):
        c, d = p.Sync(d, fb, fe, 0.0, radius)
    print(f"low texture end to end: PreSync then 4 x Sync delay {d * 1e3:.4f} ms (true {clip.delay * 1e3:.1f} ms)")
    assert abs(d - clip.delay) < 0.5e-3, d
    readouts = np.linspace(0.0, 0.022, 12)
    costs, _ = p.readout_search(readouts, d, fb, fe, 0.0005, 0.01)
    est = rsb.estimate_readout(readouts, costs)
    print(f"low texture end to end: estimated readout {est * 1e3:.3f} ms (true 11.11 ms)")
    assert abs(est - clip.readout) < 2e-3, est


def _assert_rejected(p, code, text, fn):
    before = (p.frame_table().tobytes(), p.call_counter(), p.retime_table().tobytes(), _state(p))
    with pytest.raises(rsb.RsSyncError) as e:
        fn()
    assert e.value.code == code and text in e.value.message, (e.value.code, e.value.message)
    assert (p.frame_table().tobytes(), p.call_counter(), p.retime_table().tobytes(), _state(p)) == before


def test_errors_apply_nothing(clips):
    clip, imgs = clips[(320, 240)]
    p = _problem(clip)
    _ex(p, clip, imgs, 0, 1, options=rsb.TrackOptions(cell=32))  # something to leave unchanged
    fr, ts, lens = clip.frame_ids()[:2], clip.image_ts()[:3], clip.lens()
    L = rsb.load_library()
    out = torch.empty((2 * 512, 2), dtype=torch.float64, device=DEV)
    host_out = np.empty(2 * 512)

    def call(options=rsb.TrackOptions(), points=None, counts=None, width=None, height=None, pitch=None,
             params=None, fb_out=None):
        cn = None if counts is None else np.ascontiguousarray(counts, dtype=np.uint64)
        t = np.ascontiguousarray(ts, dtype=np.float64)
        rc = L.rssync_track_frames_ex_device(
            p.h, 2, np.ascontiguousarray(fr).ctypes.data_as(rsb.c_i64_p),
            None if cn is None else cn.ctypes.data_as(rsb.C.POINTER(rsb.C.c_size_t)), t.ctypes.data_as(rsb.c_double_p),
            None if points is None else rsb.C.c_void_p(points.data_ptr()), rsb.C.c_void_p(imgs.data_ptr()),
            imgs.stride(1) if pitch is None else pitch, clip.width if width is None else width,
            clip.height if height is None else height, rsb.C.byref(rsb.Lens(*lens)),
            None if params is None else rsb.C.byref(params), rsb.C.byref(options), rsb.C.c_void_p(out.data_ptr()),
            None, None, None, fb_out, None)
        p._check(rc)

    for bad in (dict(cell=15), dict(cell=129), dict(block=4), dict(block=9), dict(block=1), dict(quality=0.0),
                dict(quality=1.5), dict(quality=float("nan")), dict(max_points=0), dict(max_points=513),
                dict(fb_max=-1.0), dict(fb_max=float("nan"))):
        _assert_rejected(p, rsb.E_INVALID, "options out of range", lambda: call(options=rsb.TrackOptions(**bad)))
    pts = torch.zeros((4, 2), dtype=torch.float64, device=DEV)
    _assert_rejected(p, rsb.E_INVALID, "both be given or both be NULL", lambda: call(points=pts))
    _assert_rejected(p, rsb.E_INVALID, "both be given or both be NULL", lambda: call(counts=[2, 2]))
    small = rsb.TrackParams(levels=1, window=5)
    _assert_rejected(p, rsb.E_INVALID, "2 * (block / 2 + 2) + 1",
                     lambda: call(width=8, params=small, options=rsb.TrackOptions(block=5)))
    _assert_rejected(p, rsb.E_INVALID, "2 * (block / 2 + 2) + 1",
                     lambda: call(height=10, params=small, options=rsb.TrackOptions(block=7)))
    _assert_rejected(p, rsb.E_INVALID, "65536 selection cells",
                     lambda: call(width=16 * 257, height=16 * 256, pitch=16 * 257, options=rsb.TrackOptions(cell=16)))
    _assert_rejected(p, rsb.E_INVALID, "an output buffer is not device memory",
                     lambda: call(fb_out=rsb.C.c_void_p(host_out.ctypes.data)))
    _assert_rejected(p, rsb.E_INVALID, "parameters out of range", lambda: call(params=rsb.TrackParams(levels=0)))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_multi_device_equals_single(clip30):
    clip, imgs = clip30
    one, multi = _problem(clip), _problem(clip, devices=[0, 1])
    opt = rsb.TrackOptions(cell=64, fb_max=1.0)
    a, b = _ex(one, clip, imgs, options=opt), _ex(multi, clip, imgs, options=opt)
    assert all(a[k].tobytes() == b[k].tobytes() for k in a)
    fb, fe = int(clip.frame_ids()[0]), int(clip.frame_ids()[-1]) + 1
    for p in (one, multi):
        p.set_rng(100, 3)
    assert one.PreSync(0.0, fb, fe, 0.002, 0.1) == multi.PreSync(0.0, fb, fe, 0.002, 0.1)
    r = [0.0, 0.008, 0.011, 0.014]
    x, y = one.readout_search(r, 0.0, fb, fe, 0.002, 0.1), multi.readout_search(r, 0.0, fb, fe, 0.002, 0.1)
    assert all(np.array_equal(u, v) for u, v in zip(x, y))
