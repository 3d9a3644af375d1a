"""The pixel -> ray front end (rssync_set_track_pixels and its device form), the rolling-shutter re-timing
(rssync_set_readout, rssync_readout_search) and the rejection of points and lenses whose undistortion
cannot be finite, against the independent restatement of tests/pixel_reference.py.

Every case runs through both forms of set_track_pixels (host arrays, torch CUDA tensors).  The stored
frames are read from the device arena and compared with the reference: timestamps, orig / pos planes,
padding lanes and the frame table with ==, rays under the reference's angle bound.  The points cover a
200-px grid of the whole image (corners, last row and column; every grid row ties in ts_a, and the rows
come in shuffled caller order), the principal point and points 5e-10 and 1e-7 from it, points outside the
image and far outside it, duplicates, and b points that are a plus a small flow.  Frame sizes sit on both
sides of the sort's powers of two, the ingest block size (256) and the 512-ray limit.  The largest bound
ratio per stage is printed at the end (run with -s)."""
import importlib

import numpy as np
import pytest

import pixel_reference as pr
import plain_reference as pl
from conftest import workload

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

synth = importlib.import_module("rs-sync_b200.synth")
W, H, R = synth.WIDTH, synth.HEIGHT, synth.READOUT
SEED = 31
LENSES = {
    "hero6": pr.Lens(*synth.LENS),
    "equidistant": pr.Lens(R, 900.0, 1150.0, 1250.5, 1100.25, 0.0, 0.0, 0.0, 0.0),
    "pincushion": pr.Lens(R, 1300.0, 1300.0, 1340.0, 1000.0, -0.02, 0.001, 0.0, 0.0),
    "strong": pr.Lens(R, 600.0, 600.0, 1355.0, 1020.0, -0.3, 0.1, -0.02, 0.01),
}
SIZES = [0, 1, 2, 31, 32, 33, 255, 256, 257, 511, 512]
IDS = np.arange(100, 100 + len(SIZES), dtype=np.int64)
RETIME = [0.0, -R, 1e-16, 2 * R]
CELL_FRAME = int(IDS[SIZES.index(256)])
LOG = pl.RatioLog()


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("\npixel reference vs engine, largest bound ratio per stage:", LOG.report())


def _cuda(x):
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64)).cuda()


def _pool(lens, rng):
    """512 points: the 200-px grid, the special points, duplicates, an offset grid, random points"""
    xs, ys = np.append(np.arange(0.0, W, 200.0), W - 1.0), np.append(np.arange(0.0, H, 200.0), H - 1.0)
    grid = np.array([(x, y) for y in ys for x in xs])
    special = np.array([(lens.cx, lens.cy), (lens.cx + 5e-10 * lens.fx, lens.cy), (lens.cx, lens.cy + 1e-7 * lens.fy),
                        (1e-9, 0.0), (-40.0, 300.0), (-1.0, -1.0), (W + 150.0, 900.0), (1200.0, H + 80.0),
                        (-3000.0, 5000.0), (1e5, 1e5)])
    grid2 = np.array([(x, y) for y in np.arange(100.0, H, 200.0) for x in np.arange(100.0, W, 200.0)])
    pts = np.concatenate([grid, special, grid[::9], special[:4], grid2])
    rand = np.column_stack([rng.uniform(-200, W + 200, 512 - len(pts)), rng.uniform(-200, H + 200, 512 - len(pts))])
    return np.concatenate([pts, rand])


class Case:
    """the frames of one lens: points (caller order), frame timestamps, and the reference frames"""

    def __init__(self, lens):
        rng = np.random.default_rng(SEED)
        pool = _pool(lens, rng)
        self.lens = lens
        self.pa, self.pb = [], []
        for n in SIZES:
            a = pool[rng.permutation(len(pool))[:n]]
            self.pa.append(a)
            self.pb.append(a + rng.normal(0.0, 1.5, a.shape))
        self.ts_a, self.ts_b = IDS / 60.0, (IDS + 1) / 60.0
        self.ref = [pr.Frame(a, b, ta, tb, lens, H) for a, b, ta, tb in zip(self.pa, self.pb, self.ts_a, self.ts_b)]

    def at(self, readout):
        return [f.retimed(a, b, ta, tb, self.lens, H, readout)
                for f, a, b, ta, tb in zip(self.ref, self.pa, self.pb, self.ts_a, self.ts_b)]

    def ingest(self, p, device, lens=None, pb=None, ids=IDS):
        pa = np.concatenate(self.pa).reshape(-1)
        pb = np.concatenate(self.pb).reshape(-1) if pb is None else pb
        if device:
            pa, pb = _cuda(pa), _cuda(pb)
        p.set_track_pixels(ids, np.asarray(SIZES, dtype=np.uint64), self.ts_a, self.ts_b, pa, pb,
                           (lens or self.lens).tuple(), H)
        return p


_CASES = {}


def case(name):
    if name not in _CASES:
        _CASES[name] = Case(LENSES[name])
    return _CASES[name]


def _problem(rsb):
    w = workload("small")
    p = rsb.SyncProblem(seed=SEED)
    p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
    return p


def _stored(p):
    """per frame id: (tiles (m, 8, 32), orig, pos) of the frame's padded range in the device arena"""
    sharded = importlib.import_module("rs-sync_b200.sharded")
    bufs, _ = sharded.device_buffers(p)
    torch.cuda.synchronize()
    host = {k: (bufs[k].cpu().numpy() if bufs[k] is not None else np.zeros(0, np.uint8)) for k in ("rays", "orig", "pos")}
    rays, orig, pos = host["rays"].view(np.float64), host["orig"].view(np.int32), host["pos"].view(np.int32)
    out = {}
    for f in p.frame_table():
        lo, m = int(f["off"]), (int(f["n"]) + 31) // 32
        out[int(f["id"])] = (rays[lo * 8:(lo + 32 * m) * 8].reshape(m, 8, 32).copy(), orig[lo:lo + 32 * m].copy(),
                             pos[lo:lo + 32 * m].copy())
    return out


def _check_stored(p, refs, stage):
    table = {int(f["id"]): f for f in p.frame_table()}
    stored = _stored(p)
    for fid, ref in zip(IDS, refs):
        fid = int(fid)
        t = table[fid]
        assert (int(t["n"]), float(t["ts_lo"]), float(t["ts_hi"])) == (ref.n, ref.ts_lo, ref.ts_hi), (stage, fid)
        tiles, orig, pos = stored[fid]
        assert np.array_equal(orig, ref.orig) and np.array_equal(pos, ref.pos), (stage, fid)
        mask = ref.ray_mask()
        assert np.array_equal(tiles[~mask], ref.tiles[~mask]), (stage, fid)  # timestamps, padding lanes
        flat = tiles.transpose(1, 0, 2).reshape(8, -1)[:, :ref.n]
        for side, und in ((slice(2, 5), ref.und_a), (slice(5, 8), ref.und_b)):
            rays = np.empty((ref.n, 3))
            rays[ref.order] = flat[side].T
            assert LOG.add("rays", pr.angle_ratio(rays, und)) <= 1.0, (stage, fid)


def _row_err(ref):
    return ref.und_a.bound + ref.und_b.bound


# ---- 1. ingest, re-timing, rows and cells ----------------------------------------------------------------
@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("name", list(LENSES))
def test_ingest_and_retime(rsb, name, device):
    c = case(name)
    p = c.ingest(_problem(rsb), device)
    assert c.ref[-1].und_a.halvings.max() > 0 and c.ref[-1].und_a.small.any() and c.ref[-1].und_a.axis.any()
    _check_stored(p, c.ref, "ingest")
    for r in RETIME:
        p.set_readout(r, int(IDS[0]), int(IDS[-1]) + 1)
        _check_stored(p, c.at(r), f"set_readout {r}")
    p.set_readout(R, int(IDS[0]), int(IDS[-1]) + 1)
    _check_stored(p, c.ref, "set_readout back")

    sr, q0, rec = p.probe_gyro()
    # problem-matrix rows (caller order) against plain_reference.rows on the reference rays
    for fid, ref in zip(IDS, c.ref):
        if ref.n < 2 or ref.n not in (33, 257, 512):
            continue
        delay = 0.021
        P = pl.rows(rec, q0, sr, delay, ref.ts_a, ref.ts_b, ref.und_a.ray.astype(np.float64),
                    ref.und_b.ray.astype(np.float64))
        bound = (pl.E + _row_err(ref))[:, None]
        assert LOG.add("rows", pl.ratio(p.probe_problem_matrix(int(fid), delay, ref.n), P.astype(np.float64),
                                        bound)) <= 1.0, fid

    # PreSync cells of one frame at the ingest readout, and through the readout search at RETIME
    delays = rsb.presync_delays(0.0, 0.02, 0.04)
    ref = c.ref[SIZES.index(256)]
    cg = p.presync_grid(CELL_FRAME, CELL_FRAME + 1, delays, call_no=6, offset_index_base=3)
    for d, delay in enumerate(delays):
        P = pl.rows(rec, q0, sr, delay, ref.ts_a, ref.ts_b, ref.und_a.ray.astype(np.float64),
                    ref.und_b.ray.astype(np.float64))
        cands = pl.presync_cell(P, pl.rng_task_key(SEED, 1, 6, 3 + d, CELL_FRAME), row_err=_row_err(ref))
        assert LOG.add("cells", pl.cell_ratio(cg[d], cands)) <= 1.0, (name, delay)
    calls = [11, 12, 13, 14]
    _, _, curves = p.readout_search(RETIME, 0.0, CELL_FRAME, CELL_FRAME + 1, 0.02, 0.04, call_nos=calls, curves=True)
    for j, r in enumerate(RETIME):
        rr = c.at(r)[SIZES.index(256)]
        for d, delay in enumerate(delays):
            P = pl.rows(rec, q0, sr, delay, rr.ts_a, rr.ts_b, rr.und_a.ray.astype(np.float64),
                        rr.und_b.ray.astype(np.float64))
            cands = pl.presync_cell(P, pl.rng_task_key(SEED, 1, calls[j], d, CELL_FRAME), row_err=_row_err(rr))
            assert LOG.add("cells", pl.cell_ratio(curves[j, d], cands)) <= 1.0, (name, r, delay)
    # the search re-times a scratch copy: the stored frames are still those of the ingest readout
    _check_stored(p, c.ref, "after readout_search")


# ---- 2. points and lenses whose undistortion cannot be finite -------------------------------------------
MSG_LENS = "set-track-pixels: bad lens profile or image height"
MSG_POINTS = "set-track-result: non-finite numbers in rays_"


def _bad_input(name, c):
    """(lens, points_b, code, message end) of a call that must be rejected"""
    hero6 = LENSES["hero6"]
    pb = np.concatenate(c.pb).reshape(-1).copy()
    if name == "far_point":  # finite, but (x - cx) / fx squared overflows: theta_ would be inf
        pb[2 * (SIZES[3] + SIZES[4] + 5)] = 1e308
        return hero6, pb, "E_NONFINITE", MSG_POINTS + "b"
    if name == "tiny_focal":  # (x - cx) / fx itself overflows for every point
        return pr.Lens(R, 1e-300, 1.0, 0.0, 0.0, 0.04, 0.0, 0.0, 0.0), pb, "E_NONFINITE", MSG_POINTS + "a"
    # k4 theta^9 overflows on (0, pi/2)
    return pr.Lens(*(hero6.tuple()[:8] + (1e308,))), pb, "E_INVALID", MSG_LENS


@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("bad", ["far_point", "tiny_focal", "lens_overflow"])
def test_rejections_leave_the_problem_unchanged(rsb, bad, device):
    c = case("hero6")
    p = c.ingest(_problem(rsb), device)
    p.set_rng(SEED, 5)
    before = (p.frame_table().tobytes(), {k: tuple(a.tobytes() for a in v) for k, v in _stored(p).items()},
              p.call_counter())
    lens, pb, code, message = _bad_input(bad, c)
    ids = np.where(np.arange(len(IDS)) % 2 == 0, IDS, IDS + 1000)  # some frames replaced, others new
    with pytest.raises(rsb.RsSyncError) as e:
        c.ingest(p, device, lens=lens, pb=pb, ids=ids)
    assert (e.value.code, e.value.message) == (getattr(rsb, code), message)
    after = (p.frame_table().tobytes(), {k: tuple(a.tobytes() for a in v) for k, v in _stored(p).items()},
             p.call_counter())
    assert after == before
    _check_stored(p, c.ref, "after rejection")
