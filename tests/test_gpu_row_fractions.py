"""Rays with rolling-shutter row fractions (rssync_set_track_row_fractions(_device), reached through
SyncProblem.set_track_row_fractions).  Every result is compared with problems fed by set_track_batch with the
timestamps formed on the host (ts = frame_ts + readout * frac): frame tables and arena tiles / orig / pos byte
for byte, PreSync / DebugPreSync / Sync and the readout search bit for bit."""
import ctypes as C

import numpy as np
import pytest

from conftest import workload
from test_gpu_readout_search import RAGGED, Frames, _arena, _cuda, _problem, _same_results, _state
from test_readout_estimate import INITIAL, RADIUS, STEP

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


class Rows:
    """ray input of some frames of a workload with per-ray row fractions: y / HEIGHT, or x / WIDTH"""

    def __init__(self, w, synth_mod, rows=None, counts=None, ids=None, columns=False):
        rows = list(range(w.n_frames)) if rows is None else list(rows)
        counts = [w.n_rays] * len(rows) if counts is None else list(counts)
        self.ids = np.asarray(w.frame_ids[rows] if ids is None else ids, dtype=np.int64)
        self.counts = np.asarray(counts, dtype=np.uint64)
        fid = w.frame_ids[rows]
        self.fts_a, self.fts_b = fid / w.fps, (fid + 1) / w.fps
        axis, size = (0, synth_mod.WIDTH) if columns else (1, synth_mod.HEIGHT)
        cat = np.concatenate
        self.qa = cat([w.px_a[r, :c, axis] / size for r, c in zip(rows, counts)])
        self.qb = cat([w.px_b[r, :c, axis] / size for r, c in zip(rows, counts)])
        self.ra = cat([w.rays_a[r, :c].reshape(-1) for r, c in zip(rows, counts)])
        self.rb = cat([w.rays_b[r, :c].reshape(-1) for r, c in zip(rows, counts)])
        self.fb, self.fe = int(self.ids.min()), int(self.ids.max()) + 1

    def per_ray(self, device):
        bufs = (self.qa, self.qb, self.ra, self.rb)
        return [_cuda(b) for b in bufs] if device else list(bufs)

    def ingest(self, p, readout, device=False):
        p.set_track_row_fractions(self.ids, self.counts, self.fts_a, self.fts_b, *self.per_ray(device), readout)
        return p

    def timestamps(self, readout):
        """the timestamps the caller would form on the host"""
        n = self.counts.astype(np.int64)
        return np.repeat(self.fts_a, n) + readout * self.qa, np.repeat(self.fts_b, n) + readout * self.qb

    def batch(self, p, readout):
        ta, tb = self.timestamps(readout)
        p.set_track_batch(self.ids, self.counts, ta, tb, self.ra, self.rb)
        return p


def _case(name, synth_mod, columns=False):
    if name == "small":
        w = workload("small")
        return w, Rows(w, synth_mod, columns=columns)
    w = workload("small", rays=512, frames=72)
    return w, Rows(w, synth_mod, counts=[RAGGED[i % len(RAGGED)] for i in range(w.n_frames)], columns=columns)


def _same_state(a, b):
    assert a.frame_table().tobytes() == b.frame_table().tobytes()
    assert _arena(a) == _arena(b)


def _reference(rsb, w, rows, readouts, calls, simplified):
    """(costs, delays, curves) of fresh set_track_batch problems at each readout, call number calls[j]"""
    delays = rsb.presync_delays(INITIAL, STEP, RADIUS)
    costs, best, curves = [], [], []
    for r, c in zip(readouts, calls):
        q = rows.batch(_problem(rsb, w, simplified), r)
        curves.append(q.presync_grid(rows.fb, rows.fe, delays, call_no=int(c)))
        q.set_rng(100, int(c))
        cost, delay = q.PreSync(INITIAL, rows.fb, rows.fe, STEP, RADIUS)
        costs.append(cost)
        best.append(delay)
    return np.array(costs), np.array(best), np.array(curves)


# ---- 1. equivalence with set_track_batch --------------------------------------------------------------
@pytest.mark.parametrize("variant", ["rows", "zero", "negative", "columns"])
@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("name", ["small", "ragged"])
def test_equals_set_track_batch(rsb, synth_mod, name, device, variant):
    w, rows = _case(name, synth_mod, columns=variant == "columns")
    R = {"rows": synth_mod.READOUT, "zero": 0.0, "negative": -0.7 * synth_mod.READOUT,
         "columns": synth_mod.READOUT}[variant]
    src = rows.ingest(_problem(rsb, w), R, device=device)
    if name == "small" and variant == "rows":  # the workload's own timestamps (synth.py forms them alike)
        assert all(np.array_equal(t, x.reshape(-1)) for t, x in zip(rows.timestamps(R), (w.ts_a, w.ts_b)))
        ref = _problem(rsb, w)
        ref.set_track_batch(w.frame_ids, rows.counts, w.ts_a, w.ts_b, w.rays_a, w.rays_b)
    else:
        ref = rows.batch(_problem(rsb, w), R)
    _same_state(src, ref)
    if variant == "rows":
        _same_results(src, ref, rows.fb, rows.fe)
    else:
        for p in (src, ref):
            p.set_rng(100, 3)
        assert src.PreSync(INITIAL, rows.fb, rows.fe, STEP, RADIUS) == ref.PreSync(INITIAL, rows.fb, rows.fe, STEP,
                                                                                   RADIUS)


# ---- 2. readout search and set_readout ------------------------------------------------------------------
@pytest.mark.parametrize("simplified", [False, True], ids=["full", "simplified"])
@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("name", ["small", "ragged"])
def test_search_and_apply(rsb, synth_mod, name, device, simplified):
    w, rows = _case(name, synth_mod)
    R = synth_mod.READOUT
    readouts = np.array([0.0, 0.5 * R, R, 1.7 * R, -0.3 * R])
    src = rows.ingest(_problem(rsb, w, simplified), R, device=device)
    src.set_rng(100, 5)
    costs, delays, curves = src.readout_search(readouts, INITIAL, rows.fb, rows.fe, STEP, RADIUS, curves=True)
    assert src.call_counter() == 5 + len(readouts)
    rc, rd, rcv = _reference(rsb, w, rows, readouts, 5 + np.arange(len(readouts)), simplified)
    assert np.array_equal(costs, rc) and np.array_equal(delays, rd) and np.array_equal(curves, rcv)
    before = _state(src)
    c2, d2 = src.readout_search(readouts, INITIAL, rows.fb, rows.fe, STEP, RADIUS, call_nos=5 + np.arange(5))
    assert np.array_equal(c2, rc) and np.array_equal(d2, rd)
    assert src.call_counter() == 5 + len(readouts) and _state(src) == before
    # applying a readout: the problem set_track_batch gives at it; back at R, the original bytes
    src.set_readout(0.0163, rows.fb, rows.fe)
    ref = rows.batch(_problem(rsb, w, simplified), 0.0163)
    _same_state(src, ref)
    if name == "small":
        _same_results(src, ref, rows.fb, rows.fe)
    src.set_readout(R, rows.fb, rows.fe)
    _same_state(src, rows.batch(_problem(rsb, w, simplified), R))


def test_search_over_pixel_and_row_frames(rsb, synth_mod):
    """one range, the first half ingested from pixels, the second from rays with row fractions"""
    w = workload("small")
    half = w.n_frames // 2
    pix, rows = Frames(w, rows=range(half)), Rows(w, synth_mod, rows=range(half, w.n_frames))
    fb, fe = pix.fb, rows.fe
    lens = lambda r: (float(r),) + tuple(synth_mod.LENS[1:])  # noqa: E731
    R = synth_mod.READOUT
    readouts = [0.0, 0.006, R, 0.016]
    src = _problem(rsb, w)
    pix.ingest(src, synth_mod, R)
    rows.ingest(src, R, device=True)
    costs, delays = src.readout_search(readouts, INITIAL, fb, fe, STEP, RADIUS, call_nos=[2] * 4)
    for j, r in enumerate(readouts):
        ref = _problem(rsb, w)
        ref.set_track_pixels(pix.ids, pix.counts, pix.ts_a, pix.ts_b, pix.pa, pix.pb, lens(r), synth_mod.HEIGHT)
        rows.batch(ref, r)
        ref.set_rng(100, 2)
        assert (costs[j], delays[j]) == ref.PreSync(INITIAL, fb, fe, STEP, RADIUS), r
    src.set_readout(0.006, fb, fe)
    ref = _problem(rsb, w)
    ref.set_track_pixels(pix.ids, pix.counts, pix.ts_a, pix.ts_b, pix.pa, pix.pb, lens(0.006), synth_mod.HEIGHT)
    _same_state(src, rows.batch(ref, 0.006))


# ---- 3. rejections --------------------------------------------------------------------------------------
@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
def test_rejections(rsb, synth_mod, device):
    w = workload("small")
    rows = Rows(w, synth_mod)
    R = synth_mod.READOUT
    p = rows.ingest(_problem(rsb, w), R)
    search = lambda: p.readout_search([0.0, R], INITIAL, rows.fb, rows.fe, STEP, RADIUS, call_nos=[1, 2])  # noqa: E731
    found = search()
    before = (_state(p), p.call_counter())
    n, F = w.n_rays, w.n_frames
    ids = rows.ids + 1000  # new frames: an applied error would show in the frame table

    def rejected(code, text, counts=rows.counts, fts=(rows.fts_a, rows.fts_b), bufs=None, readout=R):
        bufs = [b.copy() for b in (rows.qa, rows.qb, rows.ra, rows.rb)] if bufs is None else bufs
        if device:
            bufs = [_cuda(b) for b in bufs]
        with pytest.raises(rsb.RsSyncError) as e:
            p.set_track_row_fractions(ids, counts, fts[0], fts[1], *bufs, readout)
        assert e.value.code == code and text in e.value.message, e.value.message
        assert (_state(p), p.call_counter()) == before

    big = rows.counts.copy()  # the same number of rays in all, so the per-ray buffers still fit
    big[4], big[5], big[6:10] = 513, 6 * n - 513, 0
    rejected(rsb.E_INVALID, "more than 512 rays", counts=big)
    for bad in (np.nan, np.inf, -np.inf):
        rejected(rsb.E_INVALID, "set-track-row-fractions: non-finite readout", readout=bad)
    for k, which in ((0, "ts_a"), (1, "ts_b")):
        fts = [rows.fts_a.copy(), rows.fts_b.copy()]
        fts[k][7] = np.nan
        rejected(rsb.E_NONFINITE, f"non-finite numbers in {which}", fts=fts)

    def poisoned(*edits):
        """the per-ray buffers with value v at ray r of buffer k, for each (k, frame, r, v)"""
        bufs = [b.copy() for b in (rows.qa, rows.qb, rows.ra, rows.rb)]
        for k, frame, r, v in edits:
            bufs[k][(frame * n + r) * (1 if k < 2 else 3)] = v
        return bufs

    # each buffer alone (a fraction reports as its timestamp), then the buffers' and the frames' order
    for k, which in ((2, "rays_a"), (3, "rays_b"), (0, "ts_a"), (1, "ts_b")):
        for v in (np.nan, np.inf):
            rejected(rsb.E_NONFINITE, f"non-finite numbers in {which}", bufs=poisoned((k, 9, 17, v)))
    rejected(rsb.E_NONFINITE, "in rays_b", bufs=poisoned((0, 9, 3, np.nan), (3, 9, 50, np.inf), (1, 9, 0, np.nan)))
    rejected(rsb.E_NONFINITE, "in ts_b", bufs=poisoned((2, 30, 3, np.nan), (1, 12, 99, np.nan)))
    # a finite fraction whose timestamp overflows: in the product, and in the sum
    rejected(rsb.E_NONFINITE, "in ts_a", bufs=poisoned((0, 5, 1, 1e308)), readout=2.0)
    huge = rows.fts_b.copy()
    huge[F - 1] = 1e308
    rejected(rsb.E_NONFINITE, "in ts_b", fts=(rows.fts_a, huge), bufs=poisoned((1, F - 1, n - 1, 1.0)), readout=1e308)
    # the Python layer: a numpy / tensor mix
    bufs = [rows.qa, _cuda(rows.qb), rows.ra, rows.rb]
    with pytest.raises(TypeError):
        p.set_track_row_fractions(ids, rows.counts, rows.fts_a, rows.fts_b, *bufs, R)
    # the C ABI: null arguments, and (device form) memory that is not the problem's device memory
    L, cnt = p.L, rows.counts.ctypes.data_as(C.POINTER(C.c_size_t))
    fr, fa, fb = ids.ctypes.data_as(rsb.c_i64_p), rows.fts_a.ctypes.data_as(rsb.c_double_p), \
        rows.fts_b.ctypes.data_as(rsb.c_double_p)
    if device:
        t = [_cuda(b) for b in (rows.qa, rows.qb, rows.ra, rows.rb)]
        ptrs = [C.c_void_p(x.data_ptr()) for x in t]
        assert L.rssync_set_track_row_fractions_device(p.h, F, None, cnt, fa, fb, *ptrs, R, None) == rsb.E_INVALID
        assert L.rssync_set_track_row_fractions_device(p.h, F, fr, cnt, fa, None, *ptrs, R, None) == rsb.E_INVALID
        assert "set-track-row-fractions: null argument" in L.rssync_last_error(p.h).decode()
        host = [C.c_void_p(rows.qa.ctypes.data)] + ptrs[1:]
        assert L.rssync_set_track_row_fractions_device(p.h, F, fr, cnt, fa, fb, *host, R, None) == rsb.E_INVALID
        assert "not device memory" in L.rssync_last_error(p.h).decode()
        if torch.cuda.device_count() >= 2:  # a tensor on another GPU
            other = [x.to("cuda:1") for x in t]
            with pytest.raises(rsb.RsSyncError) as e:
                p.set_track_row_fractions(ids, rows.counts, rows.fts_a, rows.fts_b, *other, R)
            assert e.value.code == rsb.E_INVALID and "not device memory" in e.value.message
    else:
        dp = [b.ctypes.data_as(rsb.c_double_p) for b in (rows.qa, rows.qb, rows.ra, rows.rb)]
        for k in range(4):
            args = list(dp)
            args[k] = None
            assert L.rssync_set_track_row_fractions(p.h, F, fr, cnt, fa, fb, *args, R) == rsb.E_INVALID
        assert L.rssync_set_track_row_fractions(p.h, F, None, cnt, fa, fb, *dp, R) == rsb.E_INVALID
        assert "set-track-row-fractions: null argument" in L.rssync_last_error(p.h).decode()
    assert (_state(p), p.call_counter()) == before
    # the row-fraction plane is untouched: the search returns what it did
    found2 = search()
    assert all(np.array_equal(a, b) for a, b in zip(found, found2))


# ---- 4. duplicates and later writes ---------------------------------------------------------------------
@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
def test_duplicate_ids_keep_the_last_occurrence(rsb, synth_mod, device):
    w = workload("small", rays=512, frames=72)
    F = w.n_frames
    # frame ids 0..F-1 with ids 5 and 40 given again at the end: 5 with another size (a new arena place
    # for set_track_batch), 40 with the same padded size
    rows_all = list(range(F)) + [11, 60]
    counts = [RAGGED[i % len(RAGGED)] for i in range(F)] + [70, RAGGED[40 % len(RAGGED)]]
    ids = list(w.frame_ids[:F]) + [w.frame_ids[5], w.frame_ids[40]]
    dup = Rows(w, synth_mod, rows=rows_all, counts=counts, ids=ids)
    keep = [i for i in range(len(ids)) if i not in (5, 40)]
    last = Rows(w, synth_mod, rows=[rows_all[i] for i in keep], counts=[counts[i] for i in keep],
                ids=[ids[i] for i in keep])
    R = synth_mod.READOUT
    a = dup.ingest(_problem(rsb, w), R, device=device)
    b = last.ingest(_problem(rsb, w), R, device=device)
    _same_state(a, b)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    ra = a.readout_search([0.0, R, 0.02], INITIAL, fb, fe, STEP, RADIUS, call_nos=[1, 2, 3], curves=True)
    rb = b.readout_search([0.0, R, 0.02], INITIAL, fb, fe, STEP, RADIUS, call_nos=[1, 2, 3], curves=True)
    assert all(np.array_equal(x, y) for x, y in zip(ra, rb))


def test_later_writes_drop_the_row_fractions(rsb, synth_mod):
    w = workload("small")
    rows = Rows(w, synth_mod)
    R = synth_mod.READOUT
    p = rows.ingest(_problem(rsb, w), R, device=True)
    k = 9
    fid = int(w.frame_ids[k])
    p.SetTrackResult(fid, w.ts_a[k], w.ts_b[k], w.rays_a[k], w.rays_b[k], w.n_rays)
    for call in (lambda: p.readout_search([0.01], INITIAL, rows.fb, rows.fe, STEP, RADIUS),
                 lambda: p.set_readout(0.01, rows.fb, rows.fe)):
        with pytest.raises(rsb.RsSyncError) as e:
            call()
        assert e.value.code == rsb.E_STATE and f"frame {fid} " in e.value.message
    p.set_readout(0.01, rows.fb, fid)  # the frames before it still can
    st = p.device_state()
    dst = rsb.SyncProblem(seed=100)
    dst.adopt_state(p.frame_table(), st["arena_rays"], st["gyro_samples"], st["sample_rate"], st["first_timestamp"])
    with pytest.raises(rsb.RsSyncError) as e:
        dst.readout_search([0.01], INITIAL, rows.fb, rows.fe, STEP, RADIUS)
    assert e.value.code == rsb.E_STATE and f"frame {rows.fb} " in e.value.message


# ---- 5. borrowing ---------------------------------------------------------------------------------------
def test_device_buffers_are_borrowed(rsb, synth_mod):
    w, rows = _case("ragged", synth_mod)
    R = synth_mod.READOUT
    host = rows.ingest(_problem(rsb, w), R)
    dev = _problem(rsb, w)
    side = torch.cuda.Stream()
    pinned = [torch.from_numpy(b).pin_memory() for b in (rows.qa, rows.qb, rows.ra, rows.rb)]
    with torch.cuda.stream(side):
        # views starting one element into their allocation: 8-byte aligned only
        t = [torch.empty(x.numel() + 1, dtype=torch.float64, device="cuda")[1:] for x in pinned]
        torch.cuda._sleep(200_000_000)  # a long kernel on the producer stream, then the data
        for x, y in zip(t, pinned):
            x.copy_(y, non_blocking=True)
        dev.set_track_row_fractions(rows.ids, rows.counts, rows.fts_a, rows.fts_b, *t, R)
        for x in t:  # the caller's buffers are its own again as soon as the call returns
            x.fill_(float("nan"))
    side.synchronize()
    _same_state(dev, host)
    r = [0.0, 0.02]
    assert all(np.array_equal(x, y) for x, y in zip(
        dev.readout_search(r, INITIAL, rows.fb, rows.fe, STEP, RADIUS, call_nos=[4, 5], curves=True),
        host.readout_search(r, INITIAL, rows.fb, rows.fe, STEP, RADIUS, call_nos=[4, 5], curves=True)))


# ---- 6. several GPUs ------------------------------------------------------------------------------------
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
def test_multi_device_problem(rsb, synth_mod, device):
    w = workload("C1")
    rows = Rows(w, synth_mod)
    R = synth_mod.READOUT
    single = rows.ingest(_problem(rsb, w), R, device=device)
    multi = rows.ingest(_problem(rsb, w, devices=[0, 1]), R, device=device)
    for p in (single, multi):
        p.set_rng(100, 1)
    assert single.PreSync(INITIAL, rows.fb, rows.fe, STEP, RADIUS) == multi.PreSync(INITIAL, rows.fb, rows.fe, STEP,
                                                                                    RADIUS)
    readouts = [0.0, 0.008, 0.016]
    a = single.readout_search(readouts, INITIAL, rows.fb, rows.fe, STEP, RADIUS, call_nos=[4, 5, 6], curves=True)
    b = multi.readout_search(readouts, INITIAL, rows.fb, rows.fe, STEP, RADIUS, call_nos=[4, 5, 6], curves=True)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
