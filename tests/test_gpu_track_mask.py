"""rssync_track_frames_masked_device / SyncProblem.track_frames_ex(mask=): identity with the unmasked entry points
for a NULL and an all-ones mask (every output and the problem state); the masked selection against the
restatement (tests/mask_reference.py) bit for bit; the status rule on the caller's points and the ingest of the
status-1 pairs; a static overlay burned into every image; an independently moving object masked per image; the
rejections; a multi-device problem."""
import importlib

import numpy as np
import pytest

import mask_reference as mr
import render_reference as rr

torch = pytest.importorskip("torch")
from test_gpu_readout_search import _state  # noqa: E402
from test_gpu_track_frames import _everything, _plane, _problem, _query  # noqa: E402

pytestmark = pytest.mark.gpu
rsb = importlib.import_module("rs-sync_b200")
C = rsb.C
DEV = "cuda:0"


def _ex(p, clip, imgs, shift=None, j0=0, n=None, options=None, points=None, counts=None, mask=None, margin=None):
    n = clip.n_images - 1 - j0 if n is None else n
    r = p.track_frames_ex(clip.frame_ids()[j0:j0 + n], clip.image_ts()[j0:j0 + n + 1], imgs[j0:j0 + n + 1],
                          clip.lens(), None, options, points, counts, shift=shift, mask=mask, mask_margin=margin)
    return dict(points=r.points.cpu().numpy(), counts=r.counts, tracked=r.tracked.cpu().numpy(),
                status=r.status.cpu().numpy(), fb=r.fb_error.cpu().numpy())


def _raw(p, clip, imgs, sample, shift, mask_c, options, points=None, counts=None, frames=None, ts=None,
         pitch=None):
    """rssync_track_frames_masked_device over ctypes (mask_c: an rssync_track_mask or None for NULL)"""
    n = clip.n_images - 1
    fr = np.ascontiguousarray(clip.frame_ids() if frames is None else frames, dtype=np.int64)
    t = np.ascontiguousarray(clip.image_ts() if ts is None else ts, dtype=np.float64)
    cn = None if counts is None else np.ascontiguousarray(counts, dtype=np.uint64)
    cap = n * options.max_points if counts is None else int(cn.sum())
    out = [torch.empty(s, dtype=d, device=DEV) for s, d in (((cap, 2), torch.float64), ((cap, 2), torch.float64),
                                                            ((cap,), torch.uint8), ((cap,), torch.float64))]
    counts_out = np.zeros(fr.shape[0], dtype=np.uint64)
    rc = rsb.load_library().rssync_track_frames_masked_device(
        p.h, fr.shape[0], fr.ctypes.data_as(rsb.c_i64_p),
        None if cn is None else cn.ctypes.data_as(C.POINTER(C.c_size_t)), t.ctypes.data_as(rsb.c_double_p),
        None if points is None else C.c_void_p(points.data_ptr()), C.c_void_p(imgs.data_ptr()),
        imgs.stride(1) * imgs.element_size() if pitch is None else pitch, clip.width, clip.height, sample, shift,
        None if mask_c is None else C.byref(mask_c), C.byref(rsb.Lens(*clip.lens())), None, C.byref(options),
        C.c_void_p(out[0].data_ptr()), counts_out.ctypes.data_as(C.POINTER(C.c_size_t)),
        *[C.c_void_p(b.data_ptr()) for b in out[1:]], C.c_void_p(torch.cuda.current_stream().cuda_stream))
    p._check(rc)
    k = int(counts_out.sum())
    return dict(points=out[0][:k].cpu().numpy(), counts=counts_out.astype(np.int64), tracked=out[1][:k].cpu().numpy(),
                status=out[2][:k].cpu().numpy(), fb=out[3][:k].cpu().numpy())


def _split(x, counts):
    at = np.concatenate([[0], np.cumsum(counts)])
    return [x[at[i]:at[i + 1]] for i in range(len(counts))]


def _after(p):
    """frame table, arena and device buffers, re-timing table and row fractions"""
    return _state(p), p.retime_table().tobytes(), _plane(p)


def _assert_same(a, b, what):
    for k in a:
        assert a[k].tobytes() == b[k].tobytes(), (what, k)


def _u16(host, shift):
    return torch.from_numpy(host.astype(np.uint16) << shift).to(DEV)


def _blobs(n, h, w, seed, count=14, size=(30, 160)):
    """n seeded masks (uint8): ones with `count` zero rectangles each, some on the borders"""
    rng = np.random.default_rng(seed)
    out = np.ones((n, h, w), dtype=np.uint8)
    for j in range(n):
        for _ in range(count):
            rw, rh = rng.integers(*size, 2)
            x, y = rng.integers(-rw // 2, w - rw // 2), rng.integers(-rh // 2, h - rh // 2)
            out[j, max(0, y):y + rh, max(0, x):x + rw] = 0
    return out


@pytest.fixture(scope="module")
def clip8():
    c = rr.Clip(1001, 757, 4, delay=0.02, seed=2)
    imgs = c.render_all(DEV)
    return c, imgs, imgs.cpu().numpy()


def test_null_and_all_ones_masks_equal_unmasked(clip8):
    """mask NULL and nonzero-everywhere masks (shared, per image, expanded, padded pitch, bool, margins 0 to 63)
    give what track_frames_ex gives without a mask: every output and the problem state, 8- and 16-bit planes,
    selection and caller points, fb_max 0 and 1"""
    clip, imgs, host = clip8
    H, W, N = clip.height, clip.width, clip.n_images
    ones2 = torch.ones((H, W), dtype=torch.uint8, device=DEV)
    padded = torch.full((N, H, W + 29), 255, dtype=torch.uint8, device=DEV)[:, :, :W]
    masks = [("shared", ones2, 11), ("per image", torch.ones((N, H, W), dtype=torch.uint8, device=DEV), 0),
             ("expanded", ones2.expand(N, H, W), 63), ("padded pitch", padded, 40),
             ("bool", torch.ones((H, W), dtype=torch.bool, device=DEV), None)]
    query = _query(clip, N - 1, 40)
    counts = np.array([q.shape[0] for q in query])
    pts = torch.from_numpy(np.concatenate(query)).to(DEV)
    n_cases = 0
    for planes, shift, sample in ((imgs, None, 1), (_u16(host, 8), 8, 2)):
        for fb_max in (0.0, 1.0):
            for cell, block, caller in ((32, 5, False), (128, 7, False), (16, 3, False), (128, 5, True)):
                opt = rsb.TrackOptions(cell=cell, block=block, fb_max=fb_max)
                kw = dict(points=pts, counts=counts) if caller else {}
                ref_p = _problem(clip)
                ref = _ex(ref_p, clip, planes, shift, options=opt, **kw)
                ref_after = _after(ref_p)
                assert ref["counts"].sum() > 50
                q = _problem(clip)
                _assert_same(ref, _raw(q, clip, planes, sample, shift or 0, None, opt, **kw), "NULL")
                assert _after(q) == ref_after
                for name, m, margin in masks:
                    if caller and name not in ("shared", "padded pitch"):
                        continue
                    q = _problem(clip)
                    _assert_same(ref, _ex(q, clip, planes, shift, options=opt, mask=m, margin=margin, **kw),
                                 (name, sample, fb_max, cell))
                    assert _after(q) == ref_after, (name, sample, fb_max, cell)
                    n_cases += 1
    print(f"{n_cases} all-ones mask configurations identical to the unmasked path")


def _check_selection(got, host, masks, margin, opt, frames, what):
    for j in frames:
        ref = mr.select(host[j], mr.eligible(masks[j], margin), opt)
        pts = _split(got["points"], got["counts"])[j]
        assert pts.tobytes() == ref.tobytes(), (what, j, pts.shape, ref.shape)


def test_masked_selection_matches_restatement(clip8):
    clip, imgs, host = clip8
    masks = _blobs(clip.n_images, clip.height, clip.width, seed=5)
    m = torch.from_numpy(masks).to(DEV)
    p = _problem(clip)
    for block in (3, 5, 7):
        for cell in (16, 128):
            for margin in (0, 11, 40):
                opt = rsb.TrackOptions(cell=cell, block=block, fb_max=0.0)
                got = _ex(p, clip, imgs, options=opt, mask=m, margin=margin)
                _check_selection(got, host, masks, margin, opt, range(clip.n_images - 1), (block, cell, margin))
    # a shared mask is the per-image one repeated
    opt = rsb.TrackOptions(cell=32, fb_max=0.0)
    got = _ex(p, clip, imgs, options=opt, mask=m[1], margin=11)
    _check_selection(got, host, np.repeat(masks[1:2], clip.n_images, 0), 11, opt, range(clip.n_images - 1), "shared")


def test_masked_selection_across_chunks():
    """41 images at 2.7k with per-image masks take two pyramid chunks"""
    clip = rr.Clip(2704, 2028, 41, delay=0.02, seed=4)
    imgs = clip.render_all(DEV)
    host = imgs.cpu().numpy()
    masks = _blobs(clip.n_images, clip.height, clip.width, seed=8, count=30, size=(60, 400))
    opt = rsb.TrackOptions(cell=64, block=5, fb_max=1.0)
    got = _ex(_problem(clip), clip, imgs, options=opt, mask=torch.from_numpy(masks).to(DEV), margin=11)
    assert got["counts"].sum() > 1000
    # the selection of frames on both sides of the chunk boundary (21 images per chunk here) and the ends
    _check_selection(got, host, masks, 11, opt, (0, 1, 19, 20, 21, 22, 39), "chunks")


def test_status_rule_and_ingest(clip8):
    """caller points: tracked equals the unmasked output, statuses differ only as 1 -> 3 exactly where the
    restatement's rule says; with the backward check the status-3 points take no part in it; the problem holds
    what set_track_pixels_device gives on the status-1 pairs"""
    clip, imgs, host = clip8
    masks = _blobs(clip.n_images, clip.height, clip.width, seed=9)
    m = torch.from_numpy(masks).to(DEV)
    query = _query(clip, clip.n_images - 1, 45)
    counts = np.array([q.shape[0] for q in query])
    pts = torch.from_numpy(np.concatenate(query)).to(DEV)
    margin = 11
    elig = [mr.eligible(x, margin) for x in masks]
    fwd = rsb.TrackOptions(fb_max=0.0)
    plain = _ex(_problem(clip), clip, imgs, options=fwd, points=pts, counts=counts)
    got = _ex(_problem(clip), clip, imgs, options=fwd, points=pts, counts=counts, mask=m, margin=margin)
    assert got["tracked"].tobytes() == plain["tracked"].tobytes()
    want = np.concatenate([mr.masked_status(s, q, t, elig[j], elig[j + 1]) for j, (q, t, s) in
                           enumerate(zip(query, _split(plain["tracked"], counts), _split(plain["status"], counts)))])
    assert got["status"].tobytes() == want.tobytes()
    n3 = int(np.sum(want == 3))
    assert n3 > 50 and np.sum(want == 1) > 300, n3
    for j, (q, t, s) in enumerate(zip(query, _split(got["tracked"], counts), _split(got["status"], counts))):
        k = s == 1
        assert mr.is_eligible(elig[j], q[k]).all() and mr.is_eligible(elig[j + 1], t[k]).all()
    # the backward check: 3 where the rule says, the unmasked check's status elsewhere, NaN fb on status 3
    chk = rsb.TrackOptions(fb_max=1.0)
    plain_fb = _ex(_problem(clip), clip, imgs, options=chk, points=pts, counts=counts)
    a = _problem(clip)
    got_fb = _ex(a, clip, imgs, options=chk, points=pts, counts=counts, mask=m, margin=margin)
    assert got_fb["tracked"].tobytes() == plain_fb["tracked"].tobytes()
    three = want == 3
    assert np.array_equal(got_fb["status"] == 3, three)
    assert np.array_equal(got_fb["status"][~three], plain_fb["status"][~three])
    assert np.all(np.isnan(got_fb["fb"][three]))
    assert got_fb["fb"][~three].tobytes() == plain_fb["fb"][~three].tobytes()
    keep = got_fb["status"] == 1
    kept = np.array([int(s.sum()) for s in _split(keep, counts)])
    b = _problem(clip)
    ts = clip.image_ts()
    b.set_track_pixels(clip.frame_ids(), kept, ts[:-1], ts[1:], torch.from_numpy(got_fb["points"][keep]).to(DEV),
                       torch.from_numpy(got_fb["tracked"][keep]).to(DEV), clip.lens(), clip.height)
    assert list(a.frame_table()["n"]) == list(kept)
    fb, fe = int(clip.frame_ids()[0]), int(clip.frame_ids()[-1]) + 1
    ra, rb = _everything(a, fb, fe), _everything(b, fb, fe)
    assert [k for k in ra if ra[k] != rb[k]] == []


def _glyphs(rng, h, w):
    """a band of high-contrast 'text': 6 x 10 grids of 8-px black or white cells, 4 px apart"""
    band = np.full((h, w), 16, dtype=np.uint8)
    for x0 in range(40, w - 60, 52):
        cells = rng.integers(0, 2, (10, 6), dtype=np.uint8) * 239 + 16
        g = np.kron(cells, np.ones((8, 8), dtype=np.uint8))
        y0 = (h - g.shape[0]) // 2
        band[y0:y0 + g.shape[0], x0:x0 + g.shape[1]] = g
    return band


def _delay(p, clip):
    fb, fe = int(clip.frame_ids()[0]), int(clip.frame_ids()[-1]) + 1
    step, radius = 0.002, 0.2
    c, d = p.PreSync(0.0, fb, fe, step, radius)
    for _ in range(4):
        c, d = p.Sync(d, fb, fe, 0.0, radius)
    return d


def test_static_overlay():
    """identical glyph bands pasted into the top and bottom of every image of a 2.7k clip (true delay 37 ms):
    without a mask the selection keeps points on them; with the bands masked no kept point lies within the
    margin of them, and PreSync then 4 x Sync land within 0.1 ms of the true delay"""
    clip = rr.Clip(2704, 2028, 121, delay=0.037, seed=5)
    imgs = clip.render_all(DEV)
    rng = np.random.default_rng(21)
    band = 96
    top, bottom = (torch.from_numpy(_glyphs(rng, band, clip.width)).to(DEV) for _ in range(2))
    imgs[:, :band] = top
    imgs[:, -band:] = bottom
    mask = torch.ones((clip.height, clip.width), dtype=torch.uint8, device=DEV)
    mask[:band] = 0
    mask[-band:] = 0
    margin = 11
    opt = rsb.TrackOptions(cell=128, fb_max=1.0)
    lo, hi = band + margin, clip.height - 1 - band - margin
    out = {}
    for name, m in (("unmasked", None), ("masked", mask)):
        p = _problem(clip)
        kept_a, kept_b = [], []
        for j0 in range(0, 120, 64):
            r = _ex(p, clip, imgs, None, j0, min(64, 120 - j0), options=opt, mask=m,
                    margin=None if m is None else margin)
            k = r["status"] == 1
            kept_a.append(r["points"][k])
            kept_b.append(r["tracked"][k])
        a, b = np.concatenate(kept_a), np.concatenate(kept_b)
        out[name] = (a, b, _delay(p, clip))
    a, b, d_plain = out["unmasked"]
    in_bands = (a[:, 1] < band) | (a[:, 1] > clip.height - 1 - band)
    a, b, d_mask = out["masked"]
    print(f"static overlay: unmasked keeps {int(in_bands.sum())} points starting in the bands, delay error "
          f"{(d_plain - clip.delay) * 1e3:+.4f} ms; masked keeps {a.shape[0]} points, delay error "
          f"{(d_mask - clip.delay) * 1e3:+.4f} ms")
    assert in_bands.sum() > 100
    ya, yb = np.floor(a[:, 1] + 0.5), np.floor(b[:, 1] + 0.5)
    assert np.all((ya >= lo) & (ya <= hi) & (yb >= lo) & (yb <= hi))
    assert abs(d_mask - clip.delay) < 0.1e-3, d_mask


def test_moving_object_per_image_masks():
    """a textured square translating across the clip independently of the camera, masked per image: no kept
    point starts or ends within the margin of its footprint"""
    clip = rr.Clip(1001, 757, 9, delay=0.02, seed=3)
    imgs = clip.render_all(DEV)
    rng = np.random.default_rng(31)
    side, margin = 160, 11
    tex = torch.from_numpy(np.kron(rng.integers(0, 256, (20, 20), dtype=np.uint8), np.ones((8, 8), np.uint8))).to(DEV)
    masks = torch.ones((clip.n_images, clip.height, clip.width), dtype=torch.bool, device=DEV)
    boxes = []
    for j in range(clip.n_images):
        x0, y0 = 300 + 14 * j, 250 + 8 * j
        imgs[j, y0:y0 + side, x0:x0 + side] = tex
        masks[j, y0:y0 + side, x0:x0 + side] = False
        boxes.append((x0, y0))
    opt = rsb.TrackOptions(cell=32, fb_max=1.0)

    def near_box(pts, j):
        x0, y0 = boxes[j]
        q = mr.nearest(pts)
        return (q[:, 0] >= x0 - margin) & (q[:, 0] < x0 + side + margin) & \
               (q[:, 1] >= y0 - margin) & (q[:, 1] < y0 + side + margin)

    res = {}
    for name, m in (("unmasked", None), ("masked", masks)):
        r = _ex(_problem(clip), clip, imgs, options=opt, mask=m, margin=None if m is None else margin)
        n_on = 0
        for j, (q, t, s) in enumerate(zip(*[_split(r[k], r["counts"]) for k in ("points", "tracked", "status")])):
            k = s == 1
            n_on += int(np.sum(near_box(q[k], j) | near_box(t[k], j + 1)))
        res[name] = (n_on, int(np.sum(r["status"] == 1)))
    print(f"moving object: kept points on or next to it, unmasked {res['unmasked']}, masked {res['masked']}")
    assert res["unmasked"][0] > 20
    assert res["masked"][0] == 0 and res["masked"][1] > 300


def _assert_rejected(p, code, text, fn):
    before = (p.frame_table().tobytes(), p.call_counter(), p.retime_table().tobytes(), _state(p))
    with pytest.raises(rsb.RsSyncError) as e:
        fn()
    assert e.value.code == code and text in e.value.message, (e.value.code, e.value.message)
    assert (p.frame_table().tobytes(), p.call_counter(), p.retime_table().tobytes(), _state(p)) == before


def test_errors_apply_nothing():
    clip = rr.Clip(320, 240, 3, delay=0.02, seed=2)
    imgs = clip.render_all(DEV)
    H, W = clip.height, clip.width
    p = _problem(clip)
    mask = torch.ones((H, W), dtype=torch.uint8, device=DEV)
    _ex(p, clip, imgs, options=rsb.TrackOptions(cell=32), mask=mask)  # something to leave unchanged
    opt = rsb.TrackOptions(cell=32)
    host_mask = np.ones((H, W), dtype=np.uint8)
    tall = torch.ones((3, H, W + 8), dtype=torch.uint8, device=DEV)

    def call(ptr=mask.data_ptr(), pitch=W, stride=0, margin=11, sample=1, shift=0, planes=imgs):
        _raw(p, clip, planes, sample, shift, rsb.TrackMask(ptr, pitch, stride, margin), opt)

    _assert_rejected(p, rsb.E_INVALID, "mask is not device memory", lambda: call(ptr=host_mask.ctypes.data))
    _assert_rejected(p, rsb.E_INVALID, "mask is not device memory", lambda: call(ptr=0))
    _assert_rejected(p, rsb.E_INVALID, "mask pitch below width", lambda: call(pitch=W - 1))
    for m in (-1, 64):
        _assert_rejected(p, rsb.E_INVALID, "margin outside 0..63", lambda: call(margin=m))
    _assert_rejected(p, rsb.E_INVALID, "image_stride below height * pitch",
                     lambda: call(ptr=tall.data_ptr(), pitch=W + 8, stride=H * (W + 8) - 1))
    for s in (0, 3):
        _assert_rejected(p, rsb.E_INVALID, "sample_bytes must be 1 or 2", lambda: call(sample=s))
    _assert_rejected(p, rsb.E_INVALID, "shift 0 with 1-byte samples", lambda: call(shift=2))
    # the 16-bit checks and the ex form's, reached through the masked entry point
    wide = _u16(imgs.cpu().numpy(), 8)
    _assert_rejected(p, rsb.E_INVALID, "shift outside 0..8", lambda: call(sample=2, shift=9, planes=wide))
    _assert_rejected(p, rsb.E_INVALID, "options out of range",
                     lambda: _raw(p, clip, imgs, 1, 0, rsb.TrackMask(mask.data_ptr(), W, 0, 11),
                                  rsb.TrackOptions(cell=15)))
    # and a valid per-image stride passes
    call(ptr=tall.data_ptr(), pitch=W + 8, stride=H * (W + 8))
    # the Python front
    with pytest.raises(ValueError, match="mask must be a bool or uint8"):
        _ex(p, clip, imgs, mask=mask[:-1])
    with pytest.raises(ValueError, match="mask must be a bool or uint8"):
        _ex(p, clip, imgs, mask=mask.float())
    with pytest.raises(ValueError, match="CUDA tensor"):
        _ex(p, clip, imgs, mask=mask.cpu())
    with pytest.raises(ValueError, match="mask_margin needs a mask"):
        _ex(p, clip, imgs, margin=3)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_multi_device_equals_single(clip8):
    clip, imgs, _ = clip8
    m = torch.from_numpy(_blobs(clip.n_images, clip.height, clip.width, seed=5)).to(DEV)
    one, multi = _problem(clip), _problem(clip, devices=[0, 1])
    opt = rsb.TrackOptions(cell=64, fb_max=1.0)
    a = _ex(one, clip, imgs, options=opt, mask=m)
    b = _ex(multi, clip, imgs, options=opt, mask=m)
    _assert_same(a, b, "multi")
    fb, fe = int(clip.frame_ids()[0]), int(clip.frame_ids()[-1]) + 1
    for p in (one, multi):
        p.set_rng(100, 3)
    assert one.PreSync(0.0, fb, fe, 0.002, 0.1) == multi.PreSync(0.0, fb, fe, 0.002, 0.1)
