"""Ordering and placement of the bulk ingests that run on the problem's stream: set_track_pixels and
set_track_row_fractions (host and device forms) and track_frames_ex.  Frames set one by one before a bulk call
are older than it, and of a frame id given more than once in one call the last occurrence wins.  Each problem
is compared with one that never received the overwritten data: frame tables, arena bytes and the re-timing
table byte for byte, then PreSync or the readout search at fixed call numbers bit for bit."""
import numpy as np
import pytest

import render_reference as rr
from conftest import workload
from test_gpu_readout_search import RAGGED, Frames, _problem
from test_gpu_row_fractions import Rows, _same_state
from test_readout_estimate import INITIAL, RADIUS, STEP

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
DEV = "cuda:0"


def _batch(kind, w, synth_mod, **kw):
    """(frames of a batch, ingest(p)) of the bulk form `kind`"""
    form, where = kind.split("-")
    device = where == "device"
    if form == "pixels":
        fr = Frames(w, **kw)
        return fr, lambda p: fr.ingest(p, synth_mod, synth_mod.READOUT, device=device)
    rows = Rows(w, synth_mod, **kw)
    return rows, lambda p: rows.ingest(p, synth_mod.READOUT, device=device)


def _same(a, b):
    _same_state(a, b)
    assert a.retime_table().tobytes() == b.retime_table().tobytes()


@pytest.mark.parametrize("kind", ["pixels-host", "pixels-device", "rows-host", "rows-device"])
def test_pending_frames_go_first(rsb, synth_mod, kind):
    """every frame of the batch set one by one first, with another frame's rays of the same padded size: the
    bulk call replaces them in place, and the one-by-one data never reaches the device arena"""
    w = workload("small")
    fr, ingest = _batch(kind, w, synth_mod)
    a = _problem(rsb, w)
    F = w.n_frames
    for k in range(F):
        j = (k + 1) % F
        a.SetTrackResult(int(w.frame_ids[k]), w.ts_a[j], w.ts_b[j], w.rays_a[j], w.rays_b[j], w.n_rays)
    ingest(a)
    b = ingest(_problem(rsb, w))
    _same(a, b)
    for p in (a, b):
        p.set_rng(100, 3)
    assert a.PreSync(INITIAL, fr.fb, fr.fe, STEP, RADIUS) == b.PreSync(INITIAL, fr.fb, fr.fe, STEP, RADIUS)


@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
def test_duplicate_ids_keep_the_last_occurrence(rsb, synth_mod, device):
    w = workload("small", rays=512, frames=72)
    F = w.n_frames
    # frame ids 0..F-1 with ids 5 and 40 given again at the end: 5 with another padded size (65 -> 200 points),
    # 40 with the same padded size (64 points both times) but other points
    rows_all = list(range(F)) + [11, 60]
    counts = [RAGGED[i % len(RAGGED)] for i in range(F)] + [200, RAGGED[40 % len(RAGGED)]]
    ids = list(w.frame_ids[:F]) + [w.frame_ids[5], w.frame_ids[40]]
    dup = Frames(w, rows=rows_all, counts=counts, ids=ids)
    keep = [i for i in range(len(ids)) if i not in (5, 40)]
    last = Frames(w, rows=[rows_all[i] for i in keep], counts=[counts[i] for i in keep], ids=[ids[i] for i in keep])
    R = synth_mod.READOUT
    a = dup.ingest(_problem(rsb, w), synth_mod, R, device=device)
    b = last.ingest(_problem(rsb, w), synth_mod, R, device=device)
    _same(a, b)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    ra = a.readout_search([0.0, R, 0.02], INITIAL, fb, fe, STEP, RADIUS, call_nos=[1, 2, 3], curves=True)
    rb = b.readout_search([0.0, R, 0.02], INITIAL, fb, fe, STEP, RADIUS, call_nos=[1, 2, 3], curves=True)
    assert all(np.array_equal(x, y) for x, y in zip(ra, rb))


def test_tracker_duplicate_ids_keep_the_last_occurrence(rsb):
    from test_gpu_track_frames import _everything
    from test_gpu_track_frames import _problem as _clip_problem
    clip = rr.Clip(676, 507, 31, delay=0.031, seed=3)
    imgs = clip.render_all(DEV)
    n = clip.n_images - 1
    grid = rsb.grid_points(clip.width, clip.height, 40)
    grid = grid[(grid.min(axis=1) > 40) & (grid[:, 0] < clip.width - 40) & (grid[:, 1] < clip.height - 40)]
    # frame 20 repeats the id of frame 3 with the same padded size (40 -> 50 query points), frame 25 the id of
    # frame 7 with another one (20 -> 120)
    sizes = {3: 40, 20: 50, 7: 20, 25: 120}
    query = [grid[:sizes.get(j, 100)] for j in range(n)]
    counts = np.array([q.shape[0] for q in query])
    pts = torch.from_numpy(np.concatenate(query)).to(DEV)
    ids = clip.frame_ids()[:n].copy()
    ids[20], ids[25] = ids[3], ids[7]
    opt = rsb.TrackOptions(fb_max=0.0)

    def track(p, frames):
        r = p.track_frames_ex(frames, clip.image_ts(), imgs, clip.lens(), None, opt, pts, counts)
        return [np.asarray(x.cpu() if torch.is_tensor(x) else x) for x in (r.points, r.counts, r.tracked, r.status)]

    a = _clip_problem(clip)
    got = track(a, ids)
    # the per-point outputs stay per position: those of the same call with distinct ids
    ref = track(_clip_problem(clip), clip.frame_ids()[:n])
    assert all(x.tobytes() == y.tobytes() for x, y in zip(got, ref))
    _, _, tracked, status = got
    at = np.concatenate([[0], np.cumsum(counts)])
    kept = np.array([int(status[at[j]:at[j + 1]].astype(bool).sum()) for j in range(n)])
    pad = (kept + 31) // 32 * 32
    assert pad[3] == pad[20] and pad[7] != pad[25] and kept.min() >= 2, kept
    # the reference: the pixels form on the kept pairs of every frame but the earlier occurrences
    keep = [j for j in range(n) if j not in (3, 7)]
    sel = np.concatenate([np.arange(at[j], at[j + 1])[status[at[j]:at[j + 1]].astype(bool)] for j in keep])
    b = _clip_problem(clip)
    ts = clip.image_ts()
    b.set_track_pixels(ids[keep], kept[keep], ts[keep], ts[np.array(keep) + 1],
                       torch.from_numpy(np.concatenate(query)[sel]).to(DEV), torch.from_numpy(tracked[sel]).to(DEV),
                       clip.lens(), clip.height)
    assert a.frame_table().tobytes() == b.frame_table().tobytes()
    fb, fe = int(ids.min()), int(ids.max()) + 1
    ra, rb = _everything(a, fb, fe), _everything(b, fb, fe)
    assert [k for k in ra if ra[k] != rb[k]] == []
