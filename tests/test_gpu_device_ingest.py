"""Track input straight from GPU memory (rssync_set_track_batch_device / rssync_set_track_pixels_device,
reached through set_track_batch / set_track_pixels with torch CUDA tensors).  Every case builds one
problem through the host form and one through the device form from the same seeded workload and
compares them: frame tables with ==, arena tiles and orig / pos planes byte for byte, and every result
bit for bit."""
import importlib

import numpy as np
import pytest

from conftest import workload

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

RAGGED = [0, 1, 2, 31, 32, 33, 64, 65, 200, 511, 512]
FIELDS = ["ts_a", "ts_b", "rays_a", "rays_b"]


def _cuda(x):
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64)).cuda()


def _flat(w, rows, counts):
    """the per-ray buffers of frames `rows` of w, frame i truncated to counts[i] rays, concatenated"""
    ts_a = np.concatenate([w.ts_a[r, :c] for r, c in zip(rows, counts)])
    ts_b = np.concatenate([w.ts_b[r, :c] for r, c in zip(rows, counts)])
    ra = np.concatenate([w.rays_a[r, :c].reshape(-1) for r, c in zip(rows, counts)])
    rb = np.concatenate([w.rays_b[r, :c].reshape(-1) for r, c in zip(rows, counts)])
    return {"ts_a": ts_a, "ts_b": ts_b, "rays_a": ra, "rays_b": rb}


def _batch(p, ids, counts, bufs, device):
    b = {k: (_cuda(v) if device else v) for k, v in bufs.items()}
    p.set_track_batch(np.asarray(ids, dtype=np.int64), np.asarray(counts), b["ts_a"], b["ts_b"], b["rays_a"],
                      b["rays_b"])


def _pair(rsb, w, seed=100):
    ps = []
    for _ in range(2):
        p = rsb.SyncProblem(seed=seed)
        p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
        ps.append(p)
    return ps


def _arena(p):
    """per frame id: (tile bytes, orig bytes, pos bytes) of the frame's padded range"""
    sharded = importlib.import_module("rs-sync_b200.sharded")
    bufs, _ = sharded.device_buffers(p)
    torch.cuda.synchronize()
    host = {k: (bufs[k].cpu().numpy() if bufs[k] is not None else np.zeros(0, np.uint8)) for k in ("rays", "orig", "pos")}
    out = {}
    for f in p.frame_table():
        lo, hi = int(f["off"]), int(f["off"]) + (int(f["n"]) + 31) // 32 * 32
        out[int(f["id"])] = (host["rays"][lo * 64:hi * 64].tobytes(), host["orig"][lo * 4:hi * 4].tobytes(),
                             host["pos"][lo * 4:hi * 4].tobytes())
    return out


def _same_table(a, b):
    ta, tb = a.frame_table(), b.frame_table()
    assert ta.shape == tb.shape
    for k in ("id", "n", "ts_lo", "ts_hi"):
        assert np.array_equal(ta[k], tb[k]), k


def _same_state(a, b):
    _same_table(a, b)
    assert _arena(a) == _arena(b)
    sa, sb = a.stats(), b.stats()
    assert (sa["frames"], sa["rays"]) == (sb["frames"], sb["rays"])


def _same_results(a, b, fb, fe, probe_ids=(), full=True):
    for fid, n in probe_ids:
        assert np.array_equal(a.probe_problem_matrix(fid, 0.021, n), b.probe_problem_matrix(fid, 0.021, n))
    for p in (a, b):
        p.set_rng(100, 7)
    da, ca = a.DebugPreSync(0.0, fb, fe, 0.2, 201)
    db, cb = b.DebugPreSync(0.0, fb, fe, 0.2, 201)
    assert np.array_equal(da, db) and np.array_equal(ca, cb)
    if not full:
        return
    assert a.PreSync(0.0, fb, fe, 0.002, 0.1) == b.PreSync(0.0, fb, fe, 0.002, 0.1)
    fbs, fes = np.array([fb, fb + 20]), np.array([fb + 40, fe])
    ra, rb = a.presync_windows(0.0, fbs, fes, 0.002, 0.1), b.presync_windows(0.0, fbs, fes, 0.002, 0.1)
    assert np.array_equal(ra[0], rb[0]) and np.array_equal(ra[1], rb[1])
    assert a.Sync(0.037, fb, fb + 30, 0.0, 0.2) == b.Sync(0.037, fb, fb + 30, 0.0, 0.2)
    ini = np.array([0.036, 0.038])
    sa, sb = a.sync_batch(ini, fbs, fbs + 30, 0.0, 0.2), b.sync_batch(ini, fbs, fbs + 30, 0.0, 0.2)
    assert np.array_equal(sa[0], sb[0]) and np.array_equal(sa[1], sb[1])


# ---- 1. rays form, bit for bit ------------------------------------------------------------------
@pytest.mark.parametrize("name", ["C1", "small"])
def test_rays_form_bit_for_bit(rsb, name):
    w = workload(name)
    host, dev = _pair(rsb, w)
    rows, counts = range(w.n_frames), [w.n_rays] * w.n_frames
    bufs = _flat(w, rows, counts)
    _batch(host, w.frame_ids, counts, bufs, False)
    _batch(dev, w.frame_ids, counts, bufs, True)
    _same_state(host, dev)
    f0 = int(w.frame_ids[0])
    _same_results(host, dev, f0, int(w.frame_ids[-1]) + 1, [(f0, w.n_rays), (f0 + 17, w.n_rays)])


def test_ragged_batch_with_unusual_ids(rsb):
    """counts on both sides of every padding boundary up to 512, ids unsorted, negative and above 2^31;
    77 frames, so the host form takes its bulk path"""
    w = workload("small", rays=512, frames=77)
    counts = [RAGGED[i % len(RAGGED)] for i in range(w.n_frames)]
    rng = np.random.default_rng(5)
    ids = rng.permutation(np.concatenate([np.arange(-40, 0), 2 ** 31 - 5 + np.arange(37)]))
    # frames with fewer than 2 rays get ids outside the evaluated range (a PreSync over them is an error)
    ids = np.where(np.array(counts) < 2, -10 ** 12 - np.arange(w.n_frames), ids)
    host, dev = _pair(rsb, w)
    bufs = _flat(w, range(w.n_frames), counts)
    _batch(host, ids, counts, bufs, False)
    _batch(dev, ids, counts, bufs, True)
    _same_state(host, dev)
    good = [(int(i), c) for i, c in zip(ids, counts) if c >= 2]
    _same_results(host, dev, -40, 2 ** 31 + 40, good[:6], full=False)
    assert host.PreSync(0.0, -40, 2 ** 31 + 40, 0.002, 0.1) == dev.PreSync(0.0, -40, 2 ** 31 + 40, 0.002, 0.1)
    assert host.Sync(0.037, -40, 2 ** 31 + 40, 0.0, 0.2) == dev.Sync(0.037, -40, 2 ** 31 + 40, 0.0, 0.2)


@pytest.mark.parametrize("n", [1, 63, 64, 700])
def test_batch_sizes(rsb, n):
    w = workload("C1", frames=700, rays=40)
    host, dev = _pair(rsb, w)
    counts = [w.n_rays] * n
    bufs = _flat(w, range(n), counts)
    _batch(host, w.frame_ids[:n], counts, bufs, False)
    _batch(dev, w.frame_ids[:n], counts, bufs, True)  # a fresh problem: the arena grows from nothing
    _same_state(host, dev)
    f0 = int(w.frame_ids[0])
    _same_results(host, dev, f0, f0 + n, [(f0, w.n_rays)], full=False)


# ---- 2. pixels form ---------------------------------------------------------------------------
def test_pixels_form_bit_for_bit(rsb, synth_mod):
    w = workload("tiny", rays=130)
    counts = np.full(w.n_frames, w.n_rays)
    ta, tb = w.frame_ids / w.fps, (w.frame_ids + 1) / w.fps
    host, dev = _pair(rsb, w, seed=21)
    half = w.n_frames // 2  # two calls: the second grows the device arena, contents preserved
    for sl in (slice(0, half), slice(half, None)):
        host.set_track_pixels(w.frame_ids[sl], counts[sl], ta[sl], tb[sl], w.px_a[sl], w.px_b[sl], synth_mod.LENS,
                              synth_mod.HEIGHT)
        dev.set_track_pixels(w.frame_ids[sl], counts[sl], ta[sl], tb[sl], _cuda(w.px_a[sl].reshape(-1)),
                             _cuda(w.px_b[sl].reshape(-1)), synth_mod.LENS, synth_mod.HEIGHT)
    _same_state(host, dev)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    _same_results(host, dev, fb, fe, [(fb, w.n_rays)], full=False)
    d = np.linspace(-0.04, 0.06, 26)
    assert np.array_equal(host.presync_grid(fb, fe, d, call_no=2), dev.presync_grid(fb, fe, d, call_no=2))


# ---- 3. duplicate ids, frames set one by one around a device batch ------------------------------
def test_duplicates_and_mixing(rsb):
    w = workload("small")
    n = w.n_rays
    host, dev = _pair(rsb, w)
    ids = [int(i) for i in w.frame_ids]
    for p in (host, dev):  # one by one, still pending on the host when the batch arrives
        for r in range(10):
            p.SetTrackResult(ids[r], w.ts_a[r], w.ts_b[r], w.rays_a[r], w.rays_b[r], n)
    # frames 3, 5 replaced in place (data of other frames, same padded size), frame 7 with 20 rays (a
    # different padded size), new frames 20..59, and frame 30 given twice: the second occurrence wins
    rows = [40, 41, 42] + list(range(20, 60)) + [45]
    bid = [ids[3], ids[5], ids[7]] + ids[20:60] + [ids[30]]
    counts = [n, n, 20] + [n] * 40 + [50]
    bufs = _flat(w, rows, counts)
    _batch(host, bid, counts, bufs, False)
    _batch(dev, bid, counts, bufs, True)
    for p in (host, dev):
        p.SetTrackResult(ids[5], w.ts_a[60], w.ts_b[60], w.rays_a[60], w.rays_b[60], n)
        p.SetTrackResult(ids[62], w.ts_a[62], w.ts_b[62], w.rays_a[62], w.rays_b[62], n)
    _same_state(host, dev)
    assert dev.frame_table()["n"][list(dev.frame_table()["id"]).index(ids[30])] == 50
    _same_results(host, dev, ids[0], ids[-1] + 1, [(ids[30], 50), (ids[7], 20), (ids[3], n)])


# ---- 4. failure semantics -----------------------------------------------------------------------
@pytest.mark.parametrize("bad", [np.nan, np.inf])
@pytest.mark.parametrize("where", [0, 50, 99])
@pytest.mark.parametrize("field", FIELDS)
def test_nonfinite_rays_form(rsb, field, where, bad):
    w = workload("small", frames=100)
    w2 = workload("small", frames=100, seed=3)
    n = w.n_rays
    host, dev = _pair(rsb, w)
    counts = [n] * w.n_frames
    for p in (host, dev):
        p.set_track_batch(w.frame_ids, counts, w.ts_a, w.ts_b, w.rays_a, w.rays_b)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    delays = np.linspace(-0.05, 0.05, 11)
    before = dev.presync_grid(fb + where, fe, delays, call_no=4)
    bufs = _flat(w2, range(w.n_frames), counts)  # every frame replaced in place
    bufs[field][(where * n + 7) * (3 if field.startswith("rays") else 1) + (2 if field.startswith("rays") else 0)] = bad
    errs = []
    for p, device in ((host, False), (dev, True)):
        with pytest.raises(rsb.RsSyncError) as e:
            _batch(p, w.frame_ids, counts, bufs, device)
        errs.append((e.value.code, e.value.message))
    assert errs[0] == errs[1] and errs[0][0] == rsb.E_NONFINITE and errs[0][1].endswith(field)
    _same_state(host, dev)
    # the frames from the bad one on keep their old contents
    assert np.array_equal(dev.presync_grid(fb + where, fe, delays, call_no=4), before)
    if where:
        assert np.array_equal(host.presync_grid(fb, fb + where, delays, call_no=4),
                              dev.presync_grid(fb, fb + where, delays, call_no=4))


@pytest.mark.parametrize("where", [0, 5, 11])
@pytest.mark.parametrize("field", ["frame_ts_a", "frame_ts_b", "points_a", "points_b"])
def test_nonfinite_pixels_form(rsb, synth_mod, field, where):
    w = workload("tiny", rays=130)
    counts = np.full(w.n_frames, w.n_rays)
    args = {"frame_ts_a": w.frame_ids / w.fps, "frame_ts_b": (w.frame_ids + 1) / w.fps,
            "points_a": w.px_a.reshape(-1).copy(), "points_b": w.px_b.reshape(-1).copy()}
    ids = w.frame_ids + 1000
    host, dev = _pair(rsb, w, seed=21)
    for p in (host, dev):
        p.set_track_pixels(ids, counts, args["frame_ts_a"], args["frame_ts_b"], args["points_a"], args["points_b"],
                           synth_mod.LENS, synth_mod.HEIGHT)
    table, arena = dev.frame_table(), _arena(dev)
    args[field] = args[field].copy()
    args[field][where if field.startswith("frame") else (where * w.n_rays + 3) * 2 + 1] = np.nan
    errs = []
    for p, device in ((host, False), (dev, True)):
        pa, pb = (_cuda(args["points_a"]), _cuda(args["points_b"])) if device else (args["points_a"], args["points_b"])
        with pytest.raises(rsb.RsSyncError) as e:  # frames 1000.. replaced in place, others new
            p.set_track_pixels(w.frame_ids + 1000 + (w.frame_ids % 2) * 500, counts, args["frame_ts_a"],
                               args["frame_ts_b"], pa, pb, synth_mod.LENS, synth_mod.HEIGHT)
        errs.append((e.value.code, e.value.message))
    assert errs[0] == errs[1] and errs[0][0] == rsb.E_NONFINITE
    assert errs[0][1].endswith({"frame_ts_a": "ts_a", "frame_ts_b": "ts_b", "points_a": "rays_a",
                                "points_b": "rays_b"}[field])
    _same_state(host, dev)  # nothing applied
    assert np.array_equal(dev.frame_table(), table) and _arena(dev) == arena


# ---- 5. rejections -------------------------------------------------------------------------------
def test_rejections_leave_the_problem_unchanged(rsb):
    import ctypes as C
    w = workload("small")
    n = w.n_rays
    _, dev = _pair(rsb, w)
    dev.set_track_batch(w.frame_ids, [n] * w.n_frames, w.ts_a, w.ts_b, w.rays_a, w.rays_b)
    table, arena = dev.frame_table(), _arena(dev)
    L = dev.L
    ids = np.array([10 ** 6], dtype=np.int64)

    def call(cnt, ptrs):
        c = np.array([cnt], dtype=np.uint64)
        return L.rssync_set_track_batch_device(dev.h, 1, ids.ctypes.data_as(C.POINTER(C.c_int64)),
                                               c.ctypes.data_as(C.POINTER(C.c_size_t)), *ptrs, None)

    host_buf = np.zeros(8 * 513)
    t = torch.zeros(8 * 513, dtype=torch.float64, device="cuda")
    dptr = [C.c_void_p(t.data_ptr())] * 4
    assert call(n, [C.c_void_p(host_buf.ctypes.data)] * 4) == rsb.E_INVALID
    assert "device memory" in L.rssync_last_error(dev.h).decode()
    assert call(n, dptr[:3] + [None]) == rsb.E_INVALID
    assert call(513, dptr) == rsb.E_INVALID
    assert call(0, [None] * 4) == rsb.OK  # no rays to read: null is fine (a frame without rays)
    lens = rsb.Lens(0.01, 1000.0, 1000.0, 960.0, 540.0, 0, 0, 0, 0)
    fts = np.zeros(1)
    c = np.array([n], dtype=np.uint64)
    assert L.rssync_set_track_pixels_device(dev.h, 1, ids.ctypes.data_as(C.POINTER(C.c_int64)),
                                            c.ctypes.data_as(C.POINTER(C.c_size_t)),
                                            fts.ctypes.data_as(C.POINTER(C.c_double)),
                                            fts.ctypes.data_as(C.POINTER(C.c_double)),
                                            C.c_void_p(host_buf.ctypes.data), dptr[0], C.byref(lens), 1080.0,
                                            None) == rsb.E_INVALID
    assert call(0, [None] * 4) == rsb.OK
    tab = dev.frame_table()
    assert np.array_equal(tab[tab["id"] != 10 ** 6], table) and _arena(dev) == {**arena, 10 ** 6: _arena(dev)[10 ** 6]}
    # the Python layer: a mix of host arrays and tensors, a wrong dtype, a non-contiguous tensor
    tc = _cuda(w.ts_a[0])
    with pytest.raises(TypeError):
        dev.set_track_batch([1], [n], tc, w.ts_b[0], w.rays_a[0], w.rays_b[0])
    with pytest.raises(TypeError):
        dev.set_track_batch([1], [n], tc.float(), tc, _cuda(w.rays_a[0]), _cuda(w.rays_b[0]))
    with pytest.raises(ValueError):
        dev.set_track_batch([1], [n], tc, tc, _cuda(w.rays_a[0]).reshape(3, n).t(), _cuda(w.rays_b[0]))
    with pytest.raises(ValueError):  # fewer values than the counts give
        dev.set_track_batch([1], [n + 1], tc, tc, _cuda(w.rays_a[0]), _cuda(w.rays_b[0]))


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_buffer_on_another_device_is_rejected(rsb):
    w = workload("tiny")
    _, dev = _pair(rsb, w)
    before = dev.frame_table()
    with torch.cuda.device(1):
        b = [torch.as_tensor(np.ascontiguousarray(x.reshape(-1)), device="cuda:1")
             for x in (w.ts_a[0], w.ts_b[0], w.rays_a[0], w.rays_b[0])]
    with pytest.raises(rsb.RsSyncError) as e:
        dev.set_track_batch([1], [w.n_rays], *b)
    assert e.value.code == rsb.E_INVALID and np.array_equal(dev.frame_table(), before)


# ---- 6. ordering behind the caller's stream, and the borrow contract -----------------------------
def test_borrow_and_ordering(rsb):
    w = workload("C1")
    host, dev = _pair(rsb, w)
    counts = [w.n_rays] * w.n_frames
    bufs = _flat(w, range(w.n_frames), counts)
    _batch(host, w.frame_ids, counts, bufs, False)
    side = torch.cuda.Stream()
    pinned = {k: torch.from_numpy(v).pin_memory() for k, v in bufs.items()}
    with torch.cuda.stream(side):
        # views starting one element into their allocation: 8-byte aligned only
        t = {k: torch.empty(v.numel() + 1, dtype=torch.float64, device="cuda")[1:] for k, v in pinned.items()}
        torch.cuda._sleep(200_000_000)  # a long kernel on the producer stream, then the data
        for k in t:
            t[k].copy_(pinned[k], non_blocking=True)
        assert all(x.storage_offset() == 1 and x.is_contiguous() for x in t.values())
        dev.set_track_batch(w.frame_ids, counts, t["ts_a"], t["ts_b"], t["rays_a"], t["rays_b"])
        for x in t.values():  # the caller's buffers are its own again as soon as the call returns
            x.fill_(float("nan"))
    del t
    side.synchronize()
    _same_state(host, dev)
    f0 = int(w.frame_ids[0])
    _same_results(host, dev, f0, int(w.frame_ids[-1]) + 1, full=False)


# ---- 7. no host round trip of the data -----------------------------------------------------------
def test_bytes_over_the_bus(rsb, synth_mod):
    w = workload("C1")
    host, dev = _pair(rsb, w)
    counts = [w.n_rays] * w.n_frames
    bufs = _flat(w, range(w.n_frames), counts)
    moved = []
    for p, device in ((host, False), (dev, True)):
        p.flush()
        s0 = p.stats()
        _batch(p, w.frame_ids, counts, bufs, device)
        p.flush()
        s1 = p.stats()
        moved.append(s1["h2d_bytes"] - s0["h2d_bytes"] + s1["d2h_bytes"] - s0["d2h_bytes"])
    F, R = w.n_frames, w.n_frames * w.n_rays
    assert moved[0] >= 64 * R
    assert moved[1] <= 64 * F + 64, moved
    # pixels form: 16 more bytes per frame (the frame timestamps)
    wt = workload("tiny", rays=130)
    _, pix = _pair(rsb, wt)
    pix.flush()
    s0 = pix.stats()
    pix.set_track_pixels(wt.frame_ids, np.full(wt.n_frames, wt.n_rays), wt.frame_ids / wt.fps,
                         (wt.frame_ids + 1) / wt.fps, _cuda(wt.px_a.reshape(-1)), _cuda(wt.px_b.reshape(-1)),
                         synth_mod.LENS, synth_mod.HEIGHT)
    s1 = pix.stats()
    assert s1["h2d_bytes"] - s0["h2d_bytes"] + s1["d2h_bytes"] - s0["d2h_bytes"] <= 80 * wt.n_frames + 64


# ---- 8. several GPUs -----------------------------------------------------------------------------
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_multi_device_problem(rsb):
    w = workload("C1")
    counts = [w.n_rays] * w.n_frames
    bufs = _flat(w, range(w.n_frames), counts)
    single = rsb.SyncProblem(seed=100)
    multi = rsb.SyncProblem(seed=100, devices=[0, 1])
    for p in (single, multi):
        p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
    _batch(single, w.frame_ids, counts, bufs, False)
    with torch.cuda.device(0):
        _batch(multi, w.frame_ids, counts, bufs, True)
    _same_state(single, multi)
    f0 = int(w.frame_ids[0])
    fe = int(w.frame_ids[-1]) + 1
    for p in (single, multi):
        p.set_rng(100, 3)
    assert np.array_equal(single.DebugPreSync(0.0, f0, fe, 0.2, 201)[1], multi.DebugPreSync(0.0, f0, fe, 0.2, 201)[1])
    assert single.PreSync(0.0, f0, fe, 0.002, 0.2) == multi.PreSync(0.0, f0, fe, 0.002, 0.2)
    ini, fb = np.array([0.036, 0.037, 0.038]), np.array([f0, f0 + 100, f0 + 200])
    a, b = single.sync_batch(ini, fb, fb + 60, 0.0, 0.2), multi.sync_batch(ini, fb, fb + 60, 0.0, 0.2)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
