"""Rolling-shutter readout search and re-timing (rssync_readout_search / rssync_set_readout, reached through
SyncProblem.readout_search / set_readout).  Every result is compared with fresh problems that ingested the
same pixels with the candidate readout in the lens: (cost, delay) pairs and cost curves bit for bit, frame
tables byte for byte, arena tiles and orig / pos planes byte for byte."""
import importlib

import numpy as np
import pytest

from conftest import workload
from test_readout_estimate import INITIAL, RADIUS, READOUTS, RECOVERY_TOL, SEEDS, STEP

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

RAGGED = [2, 31, 32, 33, 64, 65, 200, 511, 512]


def _cuda(x):
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64)).cuda()


def _lens(synth_mod, readout):
    return (float(readout),) + tuple(synth_mod.LENS[1:])


class Frames:
    """pixel input of some frames of a workload: ids, counts, frame timestamps, concatenated points"""

    def __init__(self, w, rows=None, counts=None, ids=None):
        rows = list(range(w.n_frames)) if rows is None else list(rows)
        counts = [w.n_rays] * len(rows) if counts is None else list(counts)
        self.ids = np.asarray(w.frame_ids[rows] if ids is None else ids, dtype=np.int64)
        self.counts = np.asarray(counts, dtype=np.uint64)
        fid = w.frame_ids[rows]
        self.ts_a, self.ts_b = fid / w.fps, (fid + 1) / w.fps
        self.pa = np.concatenate([w.px_a[r, :c].reshape(-1) for r, c in zip(rows, counts)])
        self.pb = np.concatenate([w.px_b[r, :c].reshape(-1) for r, c in zip(rows, counts)])
        self.fb, self.fe = int(self.ids.min()), int(self.ids.max()) + 1

    def ingest(self, p, synth_mod, readout, device=False):
        pa, pb = (_cuda(self.pa), _cuda(self.pb)) if device else (self.pa, self.pb)
        p.set_track_pixels(self.ids, self.counts, self.ts_a, self.ts_b, pa, pb, _lens(synth_mod, readout),
                           synth_mod.HEIGHT)
        return p


def _problem(rsb, w, simplified=False, devices=None):
    p = rsb.SyncProblem(seed=100, devices=devices)
    p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
    p.set_loss_mode(simplified)
    return p


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


def _state(p):
    """frame table bytes, arena contents per frame, whole device buffers"""
    sharded = importlib.import_module("rs-sync_b200.sharded")
    bufs, _ = sharded.device_buffers(p)
    torch.cuda.synchronize()
    whole = tuple(bufs[k].cpu().numpy().tobytes() if bufs[k] is not None else b"" for k in
                  ("rays", "orig", "pos", "spline_records"))
    return p.frame_table().tobytes(), whole


def _reference(rsb, synth_mod, w, frames, readouts, calls, simplified):
    """(costs, delays, curves) of fresh problems ingested at each readout, PreSync at call number calls[j]"""
    delays = rsb.presync_delays(INITIAL, STEP, RADIUS)
    costs, best, curves = [], [], []
    for r, c in zip(readouts, calls):
        q = frames.ingest(_problem(rsb, w, simplified), synth_mod, r)
        curves.append(q.presync_grid(frames.fb, frames.fe, delays, call_no=int(c)))
        q.set_rng(100, int(c))
        cost, delay = q.PreSync(INITIAL, frames.fb, frames.fe, STEP, RADIUS)
        costs.append(cost)
        best.append(delay)
    return np.array(costs), np.array(best), np.array(curves)


def _case(name):
    if name == "small":
        w = workload("small")
        return w, Frames(w)
    w = workload("small", rays=512, frames=72)
    return w, Frames(w, counts=[RAGGED[i % len(RAGGED)] for i in range(w.n_frames)])


# ---- 1. search == re-ingest ---------------------------------------------------------------------------
@pytest.mark.parametrize("simplified", [False, True], ids=["full", "simplified"])
@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("name", ["small", "ragged"])
def test_search_equals_reingest(rsb, synth_mod, name, device, simplified):
    w, fr = _case(name)
    R = synth_mod.READOUT
    readouts = np.array([0.0, 0.5 * R, R, 1.7 * R, -0.3 * R])
    src = fr.ingest(_problem(rsb, w, simplified), synth_mod, R, device=device)
    src.set_rng(100, 5)
    costs, delays, curves = src.readout_search(readouts, INITIAL, fr.fb, fr.fe, STEP, RADIUS, curves=True)
    assert src.call_counter() == 5 + len(readouts)
    rc, rd, rcv = _reference(rsb, synth_mod, w, fr, readouts, 5 + np.arange(len(readouts)), simplified)
    assert np.array_equal(costs, rc) and np.array_equal(delays, rd)
    assert np.array_equal(curves, rcv)
    # without curves: the same pairs
    c2, d2 = src.readout_search(readouts, INITIAL, fr.fb, fr.fe, STEP, RADIUS, call_nos=5 + np.arange(5))
    assert np.array_equal(c2, rc) and np.array_equal(d2, rd)


# ---- 2. ties --------------------------------------------------------------------------------------------
def _tie_frames(w):
    """frames of `small` with every ray in distinct rows; at the readouts TIES the rows' r * y / rows is
    below half an ulp of the frame timestamp (all ts_a of a frame equal) or spans only a few ulps (many
    ties), while the ingest readout orders them all"""
    return Frames(w, rows=range(8))


TIES = [0.0, 1e-16, 2e-15, -2e-15]


def test_ties_search(rsb, synth_mod):
    w = workload("small")
    fr = _tie_frames(w)
    y = w.px_a[:8, :, 1]
    assert all(np.unique(row).size == row.size for row in y)
    for r in TIES[1:]:  # the crafted readouts do tie some rows, and not all of them alike
        ts = fr.ts_a[:, None] + r * (y / synth_mod.HEIGHT)
        assert any(np.unique(row).size < row.size for row in ts)
    src = fr.ingest(_problem(rsb, w), synth_mod, synth_mod.READOUT)
    costs, delays, curves = src.readout_search(TIES, INITIAL, fr.fb, fr.fe, STEP, RADIUS, call_nos=[3] * 4,
                                               curves=True)
    rc, rd, rcv = _reference(rsb, synth_mod, w, fr, TIES, [3] * 4, False)
    assert np.array_equal(costs, rc) and np.array_equal(delays, rd) and np.array_equal(curves, rcv)


@pytest.mark.parametrize("r", TIES)
def test_ties_set_readout(rsb, synth_mod, r):
    w = workload("small")
    fr = _tie_frames(w)
    src = fr.ingest(_problem(rsb, w), synth_mod, synth_mod.READOUT)
    src.set_readout(r, fr.fb, fr.fe)
    ref = fr.ingest(_problem(rsb, w), synth_mod, r)
    assert src.frame_table().tobytes() == ref.frame_table().tobytes()
    assert _arena(src) == _arena(ref)


# ---- 3. counter and side effects -----------------------------------------------------------------------
def test_counter_and_no_side_effects(rsb, synth_mod):
    w = workload("small")
    fr = Frames(w)
    src = fr.ingest(_problem(rsb, w), synth_mod, synth_mod.READOUT, device=True)
    src.set_rng(100, 11)
    before = _state(src)
    readouts = [0.004, 0.011, 0.02]
    src.readout_search(readouts, INITIAL, fr.fb, fr.fe, STEP, RADIUS, call_nos=[1, 2, 3])
    assert src.call_counter() == 11
    assert _state(src) == before
    a = src.readout_search(readouts, INITIAL, fr.fb, fr.fe, STEP, RADIUS)
    assert src.call_counter() == 14
    assert _state(src) == before
    b = src.readout_search(readouts, INITIAL, fr.fb, fr.fe, STEP, RADIUS, call_nos=[11, 12, 13])
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert src.readout_search([], INITIAL, fr.fb, fr.fe, STEP, RADIUS)[0].shape == (0,)
    assert src.call_counter() == 14


# ---- 4. set_readout -------------------------------------------------------------------------------------
def _same_results(a, b, fb, fe):
    for p in (a, b):
        p.set_rng(100, 7)
    da, ca = a.DebugPreSync(0.0, fb, fe, 0.2, 201)
    db, cb = b.DebugPreSync(0.0, fb, fe, 0.2, 201)
    assert np.array_equal(da, db) and np.array_equal(ca, cb)
    assert a.PreSync(0.0, fb, fe, 0.002, 0.1) == b.PreSync(0.0, fb, fe, 0.002, 0.1)
    assert a.Sync(0.037, fb, fb + 30, 0.0, 0.2) == b.Sync(0.037, fb, fb + 30, 0.0, 0.2)
    ini, fbs = np.array([0.036, 0.038]), np.array([fb, fb + 20])
    sa, sb = a.sync_batch(ini, fbs, fbs + 30, 0.0, 0.2), b.sync_batch(ini, fbs, fbs + 30, 0.0, 0.2)
    assert np.array_equal(sa[0], sb[0]) and np.array_equal(sa[1], sb[1])


@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
def test_set_readout_equals_reingest(rsb, synth_mod, device):
    w = workload("small")
    fr = Frames(w)
    R, R2 = synth_mod.READOUT, 0.0163
    src = fr.ingest(_problem(rsb, w), synth_mod, R, device=device)
    original = (src.frame_table().tobytes(), _arena(src))
    src.set_readout(R2, fr.fb, fr.fe)
    ref = fr.ingest(_problem(rsb, w), synth_mod, R2)
    assert src.frame_table().tobytes() == ref.frame_table().tobytes()
    assert _arena(src) == _arena(ref)
    _same_results(src, ref, fr.fb, fr.fe)
    src.set_readout(R, fr.fb, fr.fe)  # back to the ingest readout: the original bytes
    assert (src.frame_table().tobytes(), _arena(src)) == original


def test_set_readout_sub_range(rsb, synth_mod):
    w = workload("small")
    fr = Frames(w)
    R, R2 = synth_mod.READOUT, 0.004
    src = fr.ingest(_problem(rsb, w), synth_mod, R)
    before_t, before_a = src.frame_table(), _arena(src)
    lo, hi = fr.fb + 10, fr.fb + 20
    src.set_readout(R2, lo, hi)
    ref = fr.ingest(_problem(rsb, w), synth_mod, R2)
    ref_t, ref_a = ref.frame_table(), _arena(ref)
    t, a = src.frame_table(), _arena(src)
    inside = (t["id"] >= lo) & (t["id"] < hi)
    assert t[inside].tobytes() == ref_t[inside].tobytes()
    assert t[~inside].tobytes() == before_t[~inside].tobytes()
    for fid in a:
        assert a[fid] == (ref_a[fid] if lo <= fid < hi else before_a[fid]), fid
    # frames ingested later keep the lens of their own call
    w2 = workload("small", first_frame=300)
    fr2 = Frames(w2)
    fr2.ingest(src, synth_mod, R)
    fresh = fr2.ingest(_problem(rsb, w2), synth_mod, R)
    assert {k: v for k, v in _arena(src).items() if k >= 300} == _arena(fresh)


# ---- 5. rejections --------------------------------------------------------------------------------------
def _rejected(rsb, p, fb, fe, code, frame=None):
    before = (_state(p), p.call_counter())
    for call in (lambda: p.readout_search([0.01, 0.02], INITIAL, fb, fe, STEP, RADIUS),
                 lambda: p.set_readout(0.01, fb, fe)):
        with pytest.raises(rsb.RsSyncError) as e:
            call()
        assert e.value.code == code, e.value.message
        if frame is not None:
            assert f"frame {frame} " in e.value.message
        assert (_state(p), p.call_counter()) == before


@pytest.mark.parametrize("form", ["set_track", "set_track_batch", "set_track_batch_device", "overwritten"])
def test_frames_without_row_fractions_are_rejected(rsb, synth_mod, form):
    w = workload("small")
    fr = Frames(w)
    p = fr.ingest(_problem(rsb, w), synth_mod, synth_mod.READOUT)
    n = w.n_rays
    k = 9
    fid = int(w.frame_ids[k])
    if form in ("set_track", "overwritten"):  # a new frame id in range, or a pixel frame replaced
        fid = fid if form == "overwritten" else 10 ** 6
        p.SetTrackResult(fid, w.ts_a[k], w.ts_b[k], w.rays_a[k], w.rays_b[k], n)
        _rejected(rsb, p, fr.fb, max(fr.fe, fid + 1), rsb.E_STATE, fid)
        return
    # 70 frames: the host form takes its bulk path
    ids = np.arange(10 ** 6, 10 ** 6 + 70)
    rows = np.arange(70) % w.n_frames
    bufs = [w.ts_a[rows].reshape(-1), w.ts_b[rows].reshape(-1), w.rays_a[rows].reshape(-1), w.rays_b[rows].reshape(-1)]
    if form.endswith("device"):
        bufs = [_cuda(b) for b in bufs]
    p.set_track_batch(ids, [n] * 70, *bufs)
    _rejected(rsb, p, fr.fb, 10 ** 6 + 70, rsb.E_STATE, 10 ** 6)
    # the pixel frames alone still work
    p.set_readout(0.01, fr.fb, fr.fe)


def test_adopted_problem_is_rejected(rsb, synth_mod):
    w = workload("small")
    fr = Frames(w)
    src = fr.ingest(_problem(rsb, w), synth_mod, synth_mod.READOUT)
    st = src.device_state()
    dst = rsb.SyncProblem(seed=100)
    dst.adopt_state(src.frame_table(), st["arena_rays"], st["gyro_samples"], st["sample_rate"],
                    st["first_timestamp"])
    _rejected(rsb, dst, fr.fb, fr.fe, rsb.E_STATE, fr.fb)


def test_bad_readouts_are_rejected(rsb, synth_mod):
    w = workload("small")
    fr = Frames(w)
    p = fr.ingest(_problem(rsb, w), synth_mod, synth_mod.READOUT)
    before = (_state(p), p.call_counter())
    for bad in (np.nan, np.inf, -np.inf):
        with pytest.raises(rsb.RsSyncError) as e:
            p.readout_search([0.01, bad], INITIAL, fr.fb, fr.fe, STEP, RADIUS)
        assert e.value.code == rsb.E_INVALID
        with pytest.raises(rsb.RsSyncError) as e:
            p.set_readout(bad, fr.fb, fr.fe)
        assert e.value.code == rsb.E_INVALID
    r = np.array([0.01])
    c, d = np.empty(1), np.empty(1)
    assert p.L.rssync_readout_search(p.h, r.ctypes.data_as(rsb.c_double_p), -1, INITIAL, fr.fb, fr.fe, STEP, RADIUS,
                                     None, c.ctypes.data_as(rsb.c_double_p), d.ctypes.data_as(rsb.c_double_p),
                                     None) == rsb.E_INVALID
    assert (_state(p), p.call_counter()) == before
    # the pre-sync errors: bad step
    with pytest.raises(rsb.RsSyncError) as e:
        p.readout_search([0.01], INITIAL, fr.fb, fr.fe, 0.0, RADIUS)
    assert e.value.code == rsb.E_INVALID and "pre-sync" in e.value.message


# ---- 6. recovery ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", SEEDS)
def test_recovery(rsb, synth_mod, seed):
    w = workload("C1", seed=seed)
    fr = Frames(w)
    p = fr.ingest(_problem(rsb, w), synth_mod, synth_mod.READOUT, device=True)
    costs, _ = p.readout_search(READOUTS, INITIAL, fr.fb, fr.fe, STEP, RADIUS)
    v = rsb.estimate_readout(READOUTS, costs)
    assert abs(v - synth_mod.READOUT) <= RECOVERY_TOL, (seed, v, costs)
    # applying the estimate: PreSync equals a problem ingested with it
    p.set_readout(v, fr.fb, fr.fe)
    ref = fr.ingest(_problem(rsb, w), synth_mod, v)
    for q in (p, ref):
        q.set_rng(100, 0)
    assert p.PreSync(INITIAL, fr.fb, fr.fe, STEP, RADIUS) == ref.PreSync(INITIAL, fr.fb, fr.fe, STEP, RADIUS)


# ---- 7. several GPUs ------------------------------------------------------------------------------------
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_multi_device_problem(rsb, synth_mod):
    w = workload("C1")
    fr = Frames(w)
    single = fr.ingest(_problem(rsb, w), synth_mod, synth_mod.READOUT)
    multi = fr.ingest(_problem(rsb, w, devices=[0, 1]), synth_mod, synth_mod.READOUT)
    multi.PreSync(INITIAL, fr.fb, fr.fe, STEP, RADIUS)  # the replica holds the ingest readout's arena
    readouts = [0.0, 0.008, 0.016]
    a = single.readout_search(readouts, INITIAL, fr.fb, fr.fe, STEP, RADIUS, call_nos=[4, 5, 6], curves=True)
    b = multi.readout_search(readouts, INITIAL, fr.fb, fr.fe, STEP, RADIUS, call_nos=[4, 5, 6], curves=True)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    for p in (single, multi):
        p.set_readout(0.016, fr.fb, fr.fe)
        p.set_rng(100, 9)
    ref = fr.ingest(_problem(rsb, w), synth_mod, 0.016)
    ref.set_rng(100, 9)
    r = ref.PreSync(INITIAL, fr.fb, fr.fe, STEP, RADIUS)
    assert single.PreSync(INITIAL, fr.fb, fr.fe, STEP, RADIUS) == r
    assert multi.PreSync(INITIAL, fr.fb, fr.fe, STEP, RADIUS) == r  # sharded grid on the re-broadcast arena
    d = np.linspace(0.0, 0.08, 41)
    assert np.array_equal(multi.presync_grid(fr.fb, fr.fe, d, call_no=2), ref.presync_grid(fr.fb, fr.fe, d, call_no=2))
