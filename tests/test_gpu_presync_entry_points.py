"""Rejections of the PreSync entry points: PreSync (rssync_presync), presync_windows, orientation_search and
readout_search.  Each rejection is checked for its error code, its exact message and the call counter
afterwards, which tells where in the entry point the check runs.  An oversized grid (F x D > 2^34 tasks)
is built from 4096 two-ray frames and a delay grid of 5e6 offsets: it is rejected before anything the size
of the grid is reserved."""
import numpy as np
import pytest

from conftest import workload

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

INITIAL, STEP, RADIUS = 0.0, 0.005, 0.05
MSG_WINDOW = "pre-sync: search_step must be > 0 and the search window finite"
MSG_DELAYS = "pre-sync: empty or oversized delay grid"
MSG_GYRO = "pre-sync: gyro quaternions have not been set"
MSG_SIZE = "pre-sync: grid too large"
ENTRY_POINTS = ["presync", "windows", "orientation", "readout"]
# (initial, step, radius) of delay grids every entry point rejects, and the message
BAD_GRIDS = {
    "zero-step": ((INITIAL, 0.0, RADIUS), MSG_WINDOW),
    "nan-step": ((INITIAL, np.nan, RADIUS), MSG_WINDOW),
    "inf-radius": ((INITIAL, STEP, np.inf), MSG_WINDOW),
    "nan-initial": ((np.nan, STEP, RADIUS), MSG_WINDOW),
    "empty": ((INITIAL, STEP, 0.0), MSG_DELAYS),
    "oversized": ((INITIAL, 1e-9, 1.0), MSG_DELAYS),  # 2e9 offsets > 2^28
}


def _w():
    return workload("tiny", first_frame=200)  # non-negative microsecond gyro timestamps


def _problem(rsb, synth_mod, ids, counts, px_a, px_b, gyro=True, devices=None):
    """pixel frames (every entry point, the readout search included, can use them)"""
    w = _w()
    p = rsb.SyncProblem(seed=100, devices=devices)
    if gyro:
        p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
    ids = np.asarray(ids, dtype=np.int64)
    p.set_track_pixels(ids, counts, ids / w.fps, (ids + 1) / w.fps, px_a, px_b, synth_mod.LENS, synth_mod.HEIGHT)
    p.set_rng(100, 7)
    return p


def _tiny_problem(rsb, synth_mod, gyro=True, one_ray_frame=False):
    """`tiny`'s frames, optionally followed by a frame of one ray; returns (problem, fb, fe)"""
    w = _w()
    ids, counts = list(w.frame_ids), [w.n_rays] * w.n_frames
    pa, pb = w.px_a.reshape(-1), w.px_b.reshape(-1)
    if one_ray_frame:
        ids.append(int(w.frame_ids[-1]) + 1)
        counts.append(1)
        pa, pb = np.concatenate([pa, w.px_a[0, 0]]), np.concatenate([pb, w.px_b[0, 0]])
    return _problem(rsb, synth_mod, ids, counts, pa, pb, gyro), int(ids[0]), int(ids[-1]) + 1


def _call(p, entry, fb, fe, initial=INITIAL, step=STEP, radius=RADIUS):
    w = _w()
    if entry == "presync":
        return p.PreSync(initial, fb, fe, step, radius)
    if entry == "windows":
        return p.presync_windows(initial, [fb, fb], [fe, fe], step, radius)
    if entry == "orientation":
        ts = w.gyro_t0 + np.arange(w.quats.shape[0]) / w.gyro_rate
        return p.orientation_search(ts, w.omega, ["XYZ", "yXz"], initial, fb, fe, step, radius)
    return p.readout_search([0.01, 0.02], initial, fb, fe, step, radius)


def _rejected(rsb, p, entry, fb, fe, code, message, advance, **grid):
    before = p.call_counter()
    with pytest.raises(rsb.RsSyncError) as e:
        _call(p, entry, fb, fe, **grid)
    assert (e.value.code, e.value.message) == (code, message)
    assert p.call_counter() == before + advance


@pytest.mark.parametrize("grid", list(BAD_GRIDS))
@pytest.mark.parametrize("entry", ENTRY_POINTS)
def test_bad_delay_grid(rsb, synth_mod, entry, grid):
    (initial, step, radius), message = BAD_GRIDS[grid]
    p, fb, fe = _tiny_problem(rsb, synth_mod)
    _rejected(rsb, p, entry, fb, fe, rsb.E_INVALID, message, 0, initial=initial, step=step, radius=radius)
    _call(p, entry, fb, fe)  # the problem still works


# PreSync takes its call number before the grid, so its rejections there consume it
@pytest.mark.parametrize("entry,advance", [("presync", 1), ("windows", 0), ("readout", 0)])
def test_no_gyro(rsb, synth_mod, entry, advance):
    p, fb, fe = _tiny_problem(rsb, synth_mod, gyro=False)
    _rejected(rsb, p, entry, fb, fe, rsb.E_STATE, MSG_GYRO, advance)


@pytest.mark.parametrize("entry,advance", [("presync", 1), ("windows", 0), ("orientation", 0), ("readout", 0)])
def test_frame_with_one_ray(rsb, synth_mod, entry, advance):
    p, fb, fe = _tiny_problem(rsb, synth_mod, one_ray_frame=True)
    _rejected(rsb, p, entry, fb, fe, rsb.E_INVALID, f"pre-sync: frame {fe - 1} has fewer than 2 rays", advance)
    _call(p, entry, fb, fe - 1)  # without it the range is fine


# ---- oversized grid ----------------------------------------------------------------------------------
BIG_FRAMES, BIG_STEP, BIG_RADIUS = 4096, 2e-7, 0.5


def _points(rng):
    return np.column_stack([rng.uniform(100, 3900, 2 * BIG_FRAMES), rng.uniform(100, 1900, 2 * BIG_FRAMES)])


# windows advance the counter after frame selection, before the size guard; the orientation search only
# after its read-back (one device) or after its shards (several)
def _oversized(rsb, synth_mod, advance, devices=None):
    D = rsb.presync_delays(INITIAL, BIG_STEP, BIG_RADIUS).shape[0]
    assert D <= 2 ** 28 and BIG_FRAMES * D > 2 ** 34
    rng = np.random.default_rng(3)
    p = _problem(rsb, synth_mod, np.arange(BIG_FRAMES), [2] * BIG_FRAMES, _points(rng).reshape(-1),
                 _points(rng).reshape(-1), devices=devices)
    for entry in ENTRY_POINTS:
        _rejected(rsb, p, entry, 0, BIG_FRAMES, rsb.E_INVALID, MSG_SIZE, advance[entry], step=BIG_STEP,
                  radius=BIG_RADIUS)


def test_oversized_grid(rsb, synth_mod):
    _oversized(rsb, synth_mod, {"presync": 1, "windows": 2, "orientation": 0, "readout": 0})


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_oversized_grid_two_devices(rsb, synth_mod):
    _oversized(rsb, synth_mod, {"presync": 1, "windows": 2, "orientation": 2, "readout": 0}, devices=[0, 1])
