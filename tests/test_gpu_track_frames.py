"""rssync_track_frames_device / SyncProblem.track_frames on rendered rolling-shutter frames: tracked positions
against the float64 restatement (tests/track_reference.py), the ingest against set_track_pixels on the kept
pairs, batching / pitch / chunk invariance, accuracy against the true correspondences next to cv2's
Lucas-Kanade, the pipeline end to end, the rejections, and a multi-device problem."""
import importlib

import numpy as np
import pytest

import render_reference as rr
import track_reference as tr

torch = pytest.importorskip("torch")
cv2 = pytest.importorskip("cv2")
from test_gpu_readout_replicas import _wrap  # noqa: E402
from test_gpu_readout_search import _state  # noqa: E402

pytestmark = pytest.mark.gpu
rsb = importlib.import_module("rs-sync_b200")
DEV = "cuda:0"
LK_CRITERIA = (cv2.TERM_CRITERIA_COUNT | cv2.TERM_CRITERIA_EPS, 30, 0.01)
# a status may differ from the restatement's only for a point this close to a threshold: the eigenvalue
# test (relative) or the image border (pixels)
EIG_MARGIN, BORDER_MARGIN, STOP_MARGIN = 1e-3, 1e-3, 0.05


def _problem(clip, devices=None):
    p = rsb.SyncProblem(seed=100, devices=devices)
    p.SetGyroQuaternions(clip.quats, clip.quats.shape[0], clip.gyro_rate, clip.gyro_t0)
    return p


def _query(clip, n_frames, step, extra=True, seed=0):
    """per frame: the grid plus (extra) random points, points near and on the border and outside"""
    rng = np.random.default_rng([seed, clip.width, clip.height])
    W, H = clip.width, clip.height
    out = []
    for _ in range(n_frames):
        pts = [rsb.grid_points(W, H, step)]
        if extra:
            pts.append(np.stack([rng.uniform(0, W - 1, 40), rng.uniform(0, H - 1, 40)], axis=-1))
            pts.append(np.array([[0.0, 0.0], [W - 1.0, H - 1.0], [0.3, H / 2], [W - 1.2, 7.5], [-0.01, 5.0],
                                 [W - 0.99, 5.0], [-40.0, -40.0]]))
        out.append(np.concatenate(pts)[:512])
    return out


def _run(p, clip, imgs, query, j0=0, n=None, params=None):
    n = len(query) if n is None else n
    counts = np.array([q.shape[0] for q in query[j0:j0 + n]])
    pts = torch.from_numpy(np.concatenate(query[j0:j0 + n])).to(DEV)
    tracked, status = p.track_frames(clip.frame_ids()[j0:j0 + n], counts, clip.image_ts()[j0:j0 + n + 1], pts,
                                     imgs[j0:j0 + n + 1], clip.lens(), params)
    return tracked.cpu().numpy(), status.cpu().numpy().astype(bool), counts


@pytest.fixture(scope="module")
def clips():
    out = {}
    for W, H, n in ((320, 240, 4), (2704, 2028, 3), (1001, 757, 3)):
        c = rr.Clip(W, H, n, delay=0.02, seed=2)
        out[(W, H)] = (c, c.render_all(DEV))
    return out


@pytest.mark.parametrize("size", [(320, 240), (2704, 2028), (1001, 757)])
def test_positions_match_restatement(clips, size):
    clip, imgs = clips[size]
    query = _query(clip, clip.n_images - 1, max(20, clip.width // 14))
    p = _problem(clip)
    tracked, status, counts = _run(p, clip, imgs, query)
    host = imgs.cpu().numpy()
    at = np.concatenate([[0], np.cumsum(counts)])
    n_near = n_stop_near = n_both = 0
    for j, q in enumerate(query):
        ref = tr.track(host[j], host[j + 1], q)
        t, s = tracked[at[j]:at[j + 1]], status[at[j]:at[j + 1]]
        both = s & ref["status"]
        assert both.sum() >= 0.9 * q.shape[0] - 8
        err = np.hypot(*(t[both] - ref["tracked"][both]).T)
        # where an iteration's |delta| came within STOP_MARGIN of epsilon (or a level used all max_iters),
        # float32 and float64 may stop an iteration apart: such points may differ by up to 0.1 px; they are
        # counted
        stop_near = ref["stop_margin"][both] < STOP_MARGIN
        assert err[~stop_near].max() <= 1e-3, (j, err[~stop_near].max())
        assert np.all(err[stop_near] <= 0.1), (j, err[stop_near].max())
        n_stop_near += int(np.sum(err[stop_near] > 1e-3))
        n_both += int(both.sum())
        differ = s != ref["status"]
        near = (ref["eig_margin"] < EIG_MARGIN) | (np.abs(np.nan_to_num(ref["border_margin"], nan=1.0)) < BORDER_MARGIN)
        assert not np.any(differ & ~near), np.flatnonzero(differ & ~near)
        n_near += int(differ.sum())
    print(f"{size}: {n_both} points kept by both, {n_stop_near} beyond 1e-3 px next to the epsilon stop, "
          f"{n_near} status differences next to a threshold")
    assert n_near <= 2 and n_stop_near <= max(2, n_both // 50)


@pytest.fixture(scope="module")
def clip30():
    c = rr.Clip(676, 507, 31, delay=0.031, seed=3)
    return c, c.render_all(DEV)


def _kept(query, tracked, status, counts):
    at = np.concatenate([[0], np.cumsum(counts)])
    a, b, k = [], [], []
    for j, q in enumerate(query):
        s = status[at[j]:at[j + 1]]
        a.append(q[s])
        b.append(tracked[at[j]:at[j + 1]][s])
        k.append(int(s.sum()))
    return np.concatenate(a), np.concatenate(b), np.array(k)


def _plane(p):
    """the row fractions of every frame's rays (the plane's padding and spare capacity are not defined)"""
    ptr, n = p.row_fraction_plane()
    if not n:
        return b""
    plane = _wrap(ptr, n).cpu().numpy()
    return b"".join(plane[16 * int(f["off"]):16 * (int(f["off"]) + int(f["n"]))].tobytes() for f in p.frame_table())


def _everything(p, fb, fe):
    """device state, re-timing table and row fractions, then PreSync, readout search and Sync over [fb, fe)"""
    st = _state(p)
    out = dict(state=st, retime=p.retime_table().tobytes(), plane=_plane(p))
    p.set_rng(100, 7)
    out["presync"] = p.PreSync(0.0, fb, fe, 0.002, 0.1)
    out["readout"] = tuple(map(tuple, p.readout_search([0.0, 0.008, 0.011, 0.014], 0.0, fb, fe, 0.002, 0.1)))
    out["sync"] = p.Sync(out["presync"][1], fb, fe, 0.0, 0.1)
    return out


def test_ingest_identity_and_lost_frames(clip30):
    """track_frames == set_track_pixels (device form) on the kept pairs, byte for byte; a frame whose points
    are all lost and a frame without query points are ingested with 0 rays"""
    clip, imgs = clip30
    query = _query(clip, 30, 50)
    query[4] = np.array([[-3.0, 5.0], [clip.width + 2.0, 9.0]])  # all lost
    query[9] = np.zeros((0, 2))
    a = _problem(clip)
    tracked, status, counts = _run(a, clip, imgs, query)
    pa, pb, kept = _kept(query, tracked, status, counts)
    assert kept[4] == 0 and kept[9] == 0 and kept.sum() > 0.9 * counts.sum()
    b = _problem(clip)
    ts = clip.image_ts()
    b.set_track_pixels(clip.frame_ids(), kept, ts[:-1], ts[1:], torch.from_numpy(pa).to(DEV),
                       torch.from_numpy(pb).to(DEV), clip.lens(), clip.height)
    assert a.call_counter() == b.call_counter() == 0
    ft = a.frame_table()
    assert list(ft["n"]) == list(kept)
    # (PreSync rejects frames with fewer than 2 rays: the computations start after the empty frames)
    fb, fe = int(clip.frame_ids()[10]), int(clip.frame_ids()[-1]) + 1
    ra, rb = _everything(a, fb, fe), _everything(b, fb, fe)
    assert [k for k in ra if ra[k] != rb[k]] == []


def test_batching_pitch_and_chunks(clip30):
    clip, imgs = clip30
    query = _query(clip, 30, 60, extra=False)
    one = _problem(clip)
    t1, s1, _ = _run(one, clip, imgs, query)
    # batches overlapping by one image
    many = _problem(clip)
    parts = [_run(many, clip, imgs, query, j0, n) for j0, n in ((0, 7), (7, 1), (8, 22))]
    assert np.array_equal(np.concatenate([x[0] for x in parts]), t1, equal_nan=True)
    assert np.array_equal(np.concatenate([x[1] for x in parts]), s1)
    fb, fe = int(clip.frame_ids()[0]), int(clip.frame_ids()[-1]) + 1
    e1, e2 = _everything(one, fb, fe), _everything(many, fb, fe)
    assert [k for k in e1 if e1[k] != e2[k]] == []
    # strided planes: pitch > width
    wide = torch.zeros((imgs.shape[0], clip.height, clip.width + 37), dtype=torch.uint8, device=DEV)
    wide[:, :, :clip.width] = imgs
    strided = _problem(clip)
    t2, s2, _ = _run(strided, clip, wide[:, :, :clip.width], query)
    assert np.array_equal(t2, t1, equal_nan=True) and np.array_equal(s2, s1)
    e3 = _everything(strided, fb, fe)
    assert [k for k in e1 if e1[k] != e3[k]] == []


def test_several_internal_chunks():
    """2.7k planes: 256 MiB hold the pyramids of 39 images, so 41 images take two chunks; batches of 6
    frames take one each"""
    clip = rr.Clip(2704, 2028, 41, delay=0.02, seed=4)
    imgs = clip.render_all(DEV)
    per_image = sum(((2704 + (1 << l) - 1) >> l) * ((2028 + (1 << l) - 1) >> l) for l in (1, 2))
    assert (256 << 20) // (4 * per_image) < 41
    query = _query(clip, 40, 200, extra=False)
    one = _problem(clip)
    t1, s1, _ = _run(one, clip, imgs, query)
    many = _problem(clip)
    parts = [_run(many, clip, imgs, query, j0, min(6, 40 - j0)) for j0 in range(0, 40, 6)]
    assert np.array_equal(np.concatenate([x[0] for x in parts]), t1, equal_nan=True)
    assert np.array_equal(np.concatenate([x[1] for x in parts]), s1)
    assert one.frame_table().tobytes() == many.frame_table().tobytes()
    assert _state(one) == _state(many)


def _cv2_lk(a, b, pts):
    p1, st, _ = cv2.calcOpticalFlowPyrLK(a, b, pts.astype(np.float32).reshape(-1, 1, 2), None, winSize=(21, 21),
                                         maxLevel=2, criteria=LK_CRITERIA)
    return p1.reshape(-1, 2).astype(np.float64), st.ravel() == 1


def test_accuracy_against_truth_2k7(clips):
    clip, imgs = clips[(2704, 2028)]
    query = _query(clip, clip.n_images - 1, 100, extra=False)
    p = _problem(clip)
    tracked, status, counts = _run(p, clip, imgs, query)
    host = imgs.cpu().numpy()
    at = np.concatenate([[0], np.cumsum(counts)])
    ours, theirs = [], []
    for j, q in enumerate(query):
        truth = clip.true_b(j, q)
        cb, cs = _cv2_lk(host[j], host[j + 1], q)
        s = status[at[j]:at[j + 1]]
        both = s & cs
        ours.append(np.hypot(*(tracked[at[j]:at[j + 1]][both] - truth[both]).T))
        theirs.append(np.hypot(*(cb[both] - truth[both]).T))
    ours, theirs = np.concatenate(ours), np.concatenate(theirs)
    stats = {q: (float(np.percentile(ours, q)), float(np.percentile(theirs, q))) for q in (50, 90)}
    print("track_frames vs cv2 LK against the truth (px), median / p90:", stats, "points", ours.size)
    for q, (o, t) in stats.items():
        assert o <= t + 0.02, (q, o, t)


def test_end_to_end_presync_sync_readout():
    """a 2.7k clip, 121 images, true delay 37 ms, readout 11.11 ms: tracked on the 200-px grid, then PreSync,
    4 x Sync and the readout search"""
    clip = rr.Clip(2704, 2028, 121, delay=0.037, seed=5)
    imgs = clip.render_all(DEV)
    query = [rsb.grid_points(clip.width, clip.height, 200)] * 120
    p = _problem(clip)
    for j0 in range(0, 120, 64):
        n = min(64, 120 - j0)
        _run(p, clip, imgs, query, j0, n)
    fb, fe = int(clip.frame_ids()[0]), int(clip.frame_ids()[-1]) + 1
    step, radius = 0.002, 0.2
    c, d = p.PreSync(0.0, fb, fe, step, radius)
    assert abs(d - clip.delay) <= step + 1e-12, d
    for _ in range(4):
        c, d = p.Sync(d, fb, fe, 0.0, radius)
    print(f"end to end: PreSync then 4 x Sync delay {d * 1e3:.4f} ms (true {clip.delay * 1e3:.1f} ms)")
    assert abs(d - clip.delay) < 0.5e-3, d
    readouts = np.linspace(0.0, 0.022, 12)
    costs, _ = p.readout_search(readouts, d, fb, fe, 0.0005, 0.01)
    est = rsb.estimate_readout(readouts, costs)
    print(f"end to end: estimated readout {est * 1e3:.3f} ms (true 11.11 ms)")
    assert abs(est - clip.readout) < 2e-3, est
    # unpinned comparison: the reference's own front end, dense DIS sampled on the same grid
    host = imgs.cpu().numpy()
    dis = cv2.DISOpticalFlow_create(cv2.DISOPTICAL_FLOW_PRESET_MEDIUM)
    g = query[0]
    pa, pb = [], []
    for j in range(120):
        flow = dis.calc(host[j], host[j + 1], None)
        fxy = flow[np.rint(g[:, 1]).astype(int), np.rint(g[:, 0]).astype(int)]
        pa.append(g)
        pb.append(g + fxy)
    q = _problem(clip)
    ts = clip.image_ts()
    q.set_track_pixels(clip.frame_ids(), np.full(120, g.shape[0]), ts[:-1], ts[1:], np.concatenate(pa),
                       np.concatenate(pb), clip.lens(), clip.height)
    c2, d2 = q.PreSync(0.0, fb, fe, step, radius)
    for _ in range(4):
        c2, d2 = q.Sync(d2, fb, fe, 0.0, radius)
    print(f"unpinned comparison, cv2 DIS (medium) on the grid: delay {d2 * 1e3:.4f} ms")


def _assert_rejected(p, code, text, fn):
    before = (p.frame_table().tobytes(), p.call_counter(), p.retime_table().tobytes())
    with pytest.raises(rsb.RsSyncError) as e:
        fn()
    assert e.value.code == code and text in e.value.message, (e.value.code, e.value.message)
    assert (p.frame_table().tobytes(), p.call_counter(), p.retime_table().tobytes()) == before


def test_errors_apply_nothing(clips):
    clip, imgs = clips[(320, 240)]
    p = _problem(clip)
    query = _query(clip, 3, 40, extra=False)
    _run(p, clip, imgs, query[:1], 0, 1)  # something to leave unchanged
    fr, ts, lens = clip.frame_ids()[:3], clip.image_ts()[:4], clip.lens()
    counts = np.array([q.shape[0] for q in query])
    pts = torch.from_numpy(np.concatenate(query)).to(DEV)
    L = rsb.load_library()

    def call(images=imgs, points=pts, params=None, lens=lens, ts=ts, counts=counts, width=None, height=None,
             pitch=None, host_images=None):
        ip = host_images if host_images is not None else images.data_ptr()
        pp = points.data_ptr() if hasattr(points, "data_ptr") else points.ctypes.data
        cn = np.ascontiguousarray(counts, dtype=np.uint64)
        t = np.ascontiguousarray(ts, dtype=np.float64)
        rc = L.rssync_track_frames_device(
            p.h, 3, np.ascontiguousarray(fr).ctypes.data_as(rsb.c_i64_p), cn.ctypes.data_as(rsb.C.POINTER(rsb.C.c_size_t)),
            t.ctypes.data_as(rsb.c_double_p), rsb.C.c_void_p(pp), rsb.C.c_void_p(ip),
            images.stride(1) if pitch is None else pitch, clip.width if width is None else width,
            clip.height if height is None else height, rsb.C.byref(rsb.Lens(*lens)),
            None if params is None else rsb.C.byref(params), None, None, None)
        p._check(rc)

    host_img = imgs.cpu().numpy()
    _assert_rejected(p, rsb.E_INVALID, "images is not device memory", lambda: call(host_images=host_img.ctypes.data))
    host_pts = np.concatenate(query)
    _assert_rejected(p, rsb.E_INVALID, "points is not device memory", lambda: call(points=host_pts))
    _assert_rejected(p, rsb.E_INVALID, "pitch below width", lambda: call(pitch=clip.width - 1))
    _assert_rejected(p, rsb.E_INVALID, "image smaller", lambda: call(width=83, params=rsb.TrackParams(window=21)))
    _assert_rejected(p, rsb.E_INVALID, "image smaller", lambda: call(height=83))
    for bad in (dict(levels=0), dict(levels=7), dict(window=4), dict(window=22), dict(window=65),
                dict(max_iters=0), dict(max_iters=101), dict(epsilon=float("nan")), dict(epsilon=-1.0),
                dict(min_eig=float("inf"))):
        _assert_rejected(p, rsb.E_INVALID, "parameters out of range", lambda: call(params=rsb.TrackParams(**bad)))
    big = np.array([513, 1, 1])
    _assert_rejected(p, rsb.E_INVALID, "more than 512", lambda: call(counts=big))
    _assert_rejected(p, rsb.E_INVALID, "bad lens profile", lambda: call(lens=(0.011, 0.0) + tuple(lens[2:])))
    for k, side in ((0, "ts_a"), (3, "ts_b")):
        t = ts.copy()
        t[k] = np.nan
        _assert_rejected(p, rsb.E_NONFINITE, side, lambda: call(ts=t))
    nan_pts = pts.clone()
    nan_pts[5, 1] = float("nan")
    _assert_rejected(p, rsb.E_NONFINITE, "non-finite numbers in rays_a", lambda: call(points=nan_pts))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_multi_device_equals_single(clip30):
    clip, imgs = clip30
    query = _query(clip, 30, 60, extra=False)
    one, multi = _problem(clip), _problem(clip, devices=[0, 1])
    _run(one, clip, imgs, query)
    _run(multi, clip, imgs, query)
    fb, fe = int(clip.frame_ids()[0]), int(clip.frame_ids()[-1]) + 1
    for p in (one, multi):
        p.set_rng(100, 3)
    assert one.PreSync(0.0, fb, fe, 0.002, 0.1) == multi.PreSync(0.0, fb, fe, 0.002, 0.1)
    r = [0.0, 0.008, 0.011, 0.014]
    a, b = one.readout_search(r, 0.0, fb, fe, 0.002, 0.1), multi.readout_search(r, 0.0, fb, fe, 0.002, 0.1)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
