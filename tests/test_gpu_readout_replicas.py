"""The rolling-shutter readout search on replicas: a problem that adopted another's state and row fractions
(rssync_adopt_row_fractions), a multi-device problem that shards the readouts over its devices, and the
one-process-per-GPU form (sharded.replicate_row_fractions + readout_search_sharded).  Every result is
compared bit for bit with the single-device search of a problem that ingested the frames itself."""
import importlib
import itertools
import os
import sys

import numpy as np
import pytest

import plain_reference as ref
from conftest import ROOT, workload
from test_gpu_readout_search import RAGGED, Frames, _arena, _problem, _state
from test_gpu_row_fractions import Rows
from test_readout_estimate import INITIAL, RADIUS, STEP

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

N_GPUS = torch.cuda.device_count() if torch.cuda.is_available() else 0
needs2 = pytest.mark.skipif(N_GPUS < 2, reason="needs 2 GPUs")
RAGGED_BASE = 100000  # ids of the ragged row-fraction frames, after C1's


def _sharded():
    return importlib.import_module("rs-sync_b200.sharded")


def _wrap(ptr, nbytes):
    return torch.as_tensor(_sharded()._DevicePtr(ptr, nbytes), device="cuda")


class Source:
    """C1 from pixels and a ragged 2..512-ray batch from row fractions, in one problem"""

    def __init__(self, rsb, synth_mod, simplified=False, device=False):
        self.w = workload("C1")
        wr = workload("small", rays=512, frames=72)
        self.pix = Frames(self.w)
        counts = [RAGGED[i % len(RAGGED)] for i in range(wr.n_frames)]
        self.rows = Rows(wr, synth_mod, counts=counts, ids=RAGGED_BASE + np.arange(wr.n_frames))
        self.fb, self.fe = self.pix.fb, int(self.rows.ids.max()) + 1
        self.synth_mod, self.simplified = synth_mod, simplified
        self.p = self.ingest(_problem(rsb, self.w, simplified), synth_mod.READOUT, device)

    def ingest(self, p, readout, device=False):
        self.pix.ingest(p, self.synth_mod, readout, device=device)
        self.rows.ingest(p, readout, device=device)
        return p


def _adopt(rsb, src, simplified=False, stream=None):
    """a problem on the same device that adopts src's state and row fractions; device-to-device copies stand
    in for the broadcasts.  stream: the side stream that fills the plane (announced with expect_chunk)"""
    sh = _sharded()
    bufs, st = sh.device_buffers(src)
    dst = rsb.SyncProblem(seed=100)
    dst.set_loss_mode(simplified)
    dst.adopt_state(src.frame_table(), st["arena_rays"], st["gyro_samples"], st["sample_rate"], st["first_timestamp"])
    dbufs, _ = sh.device_buffers(dst)
    for k in ("rays", "orig", "pos", "spline_records"):
        dbufs[k].copy_(bufs[k])
    torch.cuda.synchronize()
    dst.adopt_row_fractions(src.retime_table())
    sp, sn = src.row_fraction_plane()
    dp, dn = dst.row_fraction_plane()
    assert sn == dn == 16 * st["arena_rays"] and sp and dp
    if stream is None:
        _wrap(dp, dn).copy_(_wrap(sp, sn))
        torch.cuda.synchronize()
    return dst, _wrap(sp, sn), _wrap(dp, dn)


READOUTS = np.array([0.0, 0.004, 0.0123, 0.02, -0.003])


def _search(p, fb, fe, readouts=READOUTS, call_nos=None, counter=11):
    p.set_rng(100, counter)
    out = p.readout_search(readouts, INITIAL, fb, fe, STEP, RADIUS, call_nos=call_nos, curves=True)
    return out, p.call_counter()


def _equal(a, b):
    (ra, ca), (rb, cb) = a, b
    assert all(np.array_equal(x, y) for x, y in zip(ra, rb)) and ca == cb


# ---- 1. adoption (one GPU) ------------------------------------------------------------------------------
@pytest.mark.parametrize("simplified", [False, True], ids=["full", "simplified"])
@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
def test_adopted_problem_searches_and_applies(rsb, synth_mod, simplified, device):
    s = Source(rsb, synth_mod, simplified, device)
    src = s.p
    dst, _, _ = _adopt(rsb, src, simplified)
    assert np.array_equal(dst.retime_table(), src.retime_table())
    assert len(dst.retime_table()) == s.pix.ids.size + s.rows.ids.size
    for call_nos in (None, 3 + np.arange(len(READOUTS))):
        _equal(_search(dst, s.fb, s.fe, call_nos=call_nos), _search(src, s.fb, s.fe, call_nos=call_nos))
    # the pixel part alone and the row-fraction part alone
    _equal(_search(dst, s.pix.fb, s.pix.fe), _search(src, s.pix.fb, s.pix.fe))
    _equal(_search(dst, s.rows.fb, s.rows.fe), _search(src, s.rows.fb, s.rows.fe))
    # set_readout, then PreSync: a fresh ingest at that readout
    R2 = 0.0163
    dst.set_readout(R2, s.fb, s.fe)
    fresh = s.ingest(_problem(rsb, s.w, simplified), R2)
    for p in (dst, fresh):
        p.set_rng(100, 2)
    assert dst.PreSync(INITIAL, s.fb, s.fe, STEP, RADIUS) == fresh.PreSync(INITIAL, s.fb, s.fe, STEP, RADIUS)
    # arena and frame table byte for byte, as the source holds them after the same set_readout
    src.set_readout(R2, s.fb, s.fe)
    assert dst.frame_table().tobytes() == src.frame_table().tobytes() == fresh.frame_table().tobytes()
    assert _arena(dst) == _arena(src) == _arena(fresh)


def test_plane_filled_on_a_busy_stream(rsb, synth_mod):
    """the plane arrives late on a side stream announced with expect_chunk; the source's plane is
    overwritten right after the copy: the receiver's search waits for the copy and sees the source's data"""
    s = Source(rsb, synth_mod)
    want = _search(s.p, s.fb, s.fe, call_nos=1 + np.arange(len(READOUTS)))
    side = torch.cuda.Stream()
    dst, splane, dplane = _adopt(rsb, s.p, stream=side)
    dplane.zero_()
    torch.cuda.synchronize()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)
        dplane.copy_(splane)
        dst.expect_chunk(0, dplane.numel() // 16, side.cuda_stream)
        splane.fill_(255)  # NaN in every double of the source's plane
    _equal(_search(dst, s.fb, s.fe, call_nos=1 + np.arange(len(READOUTS))), want)
    side.synchronize()
    # the second path that reads the plane, on a fresh receiver: set_readout orders itself the same way
    s2 = Source(rsb, synth_mod)
    dst2, splane2, dplane2 = _adopt(rsb, s2.p, stream=side)
    dplane2.zero_()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)
        dplane2.copy_(splane2)
        dst2.expect_chunk(0, dplane2.numel() // 16, side.cuda_stream)
    dst2.set_readout(0.0163, s2.fb, s2.fe)
    s2.p.set_readout(0.0163, s2.fb, s2.fe)
    assert _arena(dst2) == _arena(s2.p)


def test_adoption_rejections(rsb, synth_mod):
    s = Source(rsb, synth_mod)
    table = s.p.retime_table()
    # a problem that ingested its own frames
    with pytest.raises(rsb.RsSyncError) as e:
        s.p.adopt_row_fractions(table)
    assert e.value.code == rsb.E_STATE
    dst, _, _ = _adopt(rsb, s.p)
    want = _search(dst, s.fb, s.fe, call_nos=np.arange(len(READOUTS)))
    before = (dst.retime_table().tobytes(), dst.call_counter(), _state(dst))

    def unchanged():
        assert (dst.retime_table().tobytes(), dst.call_counter(), _state(dst)) == before
        _equal(_search(dst, s.fb, s.fe, call_nos=np.arange(len(READOUTS))), want)
        dst.set_rng(100, before[1])

    unknown = table.copy()
    unknown["id"][3] = 123456789
    repeated = np.concatenate([table, table[5:6]])
    nan = table.copy()
    nan["frame_ts_b"][7] = np.nan
    for bad, text in ((unknown, "not in the adopted frame table"), (repeated, "given more than once"),
                      (nan, "non-finite frame timestamp")):
        with pytest.raises(rsb.RsSyncError) as e:
            dst.adopt_row_fractions(bad)
        assert e.value.code == rsb.E_INVALID and text in e.value.message
        unchanged()
    assert rsb.load_library().rssync_adopt_row_fractions(dst.h, None, 3) == rsb.E_INVALID
    unchanged()
    # after a Set* call that follows the adoption
    dst.SetGyroQuaternions(s.w.quats, s.w.quats.shape[0], s.w.gyro_rate, s.w.gyro_t0)
    with pytest.raises(rsb.RsSyncError) as e:
        dst.adopt_row_fractions(table)
    assert e.value.code == rsb.E_STATE


def test_adoption_without_row_fractions_and_overwrites(rsb, synth_mod):
    s = Source(rsb, synth_mod)
    sh = _sharded()
    bufs, st = sh.device_buffers(s.p)
    dst = rsb.SyncProblem(seed=100)
    dst.adopt_state(s.p.frame_table(), st["arena_rays"], st["gyro_samples"], st["sample_rate"], st["first_timestamp"])
    dbufs, _ = sh.device_buffers(dst)
    for k in ("rays", "orig", "pos", "spline_records"):
        dbufs[k].copy_(bufs[k])
    torch.cuda.synchronize()
    assert dst.retime_table().size == 0 and dst.row_fraction_plane() == (0, 0)
    counter = dst.call_counter()
    with pytest.raises(rsb.RsSyncError) as e:
        dst.readout_search(READOUTS, INITIAL, s.fb, s.fe, STEP, RADIUS)
    assert e.value.code == rsb.E_STATE and dst.call_counter() == counter
    # with the row fractions, a rays-form overwrite of an adopted frame drops it from the table
    dst2, _, _ = _adopt(rsb, s.p)
    w, fid = s.w, int(s.pix.ids[4])
    dst2.set_track_batch(np.array([fid]), np.array([w.n_rays], dtype=np.uint64), w.ts_a[4], w.ts_b[4],
                         w.rays_a[4].reshape(-1), w.rays_b[4].reshape(-1))
    ids = dst2.retime_table()["id"]
    assert fid not in ids and ids.size == s.pix.ids.size + s.rows.ids.size - 1
    # and a later adopt_state drops them all
    dst2.adopt_state(s.p.frame_table(), st["arena_rays"], st["gyro_samples"], st["sample_rate"], st["first_timestamp"])
    assert dst2.retime_table().size == 0


# ---- 2. several GPUs behind one problem -----------------------------------------------------------------
def _pair(rsb, w, simplified=False):
    return _problem(rsb, w, simplified), _problem(rsb, w, simplified, devices=list(range(N_GPUS)))


@needs2
@pytest.mark.parametrize("simplified", [False, True], ids=["full", "simplified"])
def test_multi_device_search_equals_one_device(rsb, synth_mod, simplified):
    w = workload("small")
    half = w.n_frames // 2
    pix, rows = Frames(w, rows=range(half)), Rows(w, synth_mod, rows=range(half, w.n_frames))
    one, many = _pair(rsb, w, simplified)
    for p in (one, many):
        pix.ingest(p, synth_mod, synth_mod.READOUT)
        rows.ingest(p, synth_mod.READOUT, device=True)
    G = N_GPUS
    rng = np.random.default_rng(3)
    for n in sorted({1, 2, G - 1, G, G + 1, 11} - {0}):
        readouts = rng.uniform(-0.005, 0.025, n)
        for fb, fe in ((pix.fb, pix.fe), (rows.fb, rows.fe), (pix.fb, rows.fe)):
            for call_nos in (None, 50 + 3 * np.arange(n)):
                _equal(_search(many, fb, fe, readouts, call_nos), _search(one, fb, fe, readouts, call_nos))
                assert many.stats()["last_grid_tasks"] == one.stats()["last_grid_tasks"]
                assert many.stats()["last_grid_exact_tasks"] == one.stats()["last_grid_exact_tasks"]


def _error(rsb, p, *args, **kw):
    """(code, message, counter advance) of a search that must fail"""
    counter = p.call_counter()
    with pytest.raises(rsb.RsSyncError) as e:
        p.readout_search(*args, **kw)
    return e.value.code, e.value.message, p.call_counter() - counter


@needs2
def test_multi_device_errors_equal_one_device(rsb, synth_mod):
    w = workload("small")
    fr = Frames(w)
    one, many = _pair(rsb, w)
    for p in (one, many):
        fr.ingest(p, synth_mod, synth_mod.READOUT)
        # a rays-form frame inside the range
        p.set_track_batch(np.array([fr.fe + 1]), np.array([w.n_rays], dtype=np.uint64), w.ts_a[0], w.ts_b[0],
                          w.rays_a[0].reshape(-1), w.rays_b[0].reshape(-1))
    args = (READOUTS, INITIAL, fr.fb, fr.fe + 2, STEP, RADIUS)
    a, b = _error(rsb, one, *args), _error(rsb, many, *args)
    assert a == b and a[0] == rsb.E_STATE and a[2] == 0


def _panic_frame(w, call_no, n):
    """the pixels of w's first frame with the ray pair the estimator draws first (call call_no, delay 0)
    made equal: that hypothesis is exactly 0 and gives the reference's panic "pre-sync: non-finite r" at
    every readout (equal pixels are re-timed alike)"""
    fid = int(w.frame_ids[0])
    a, b = ref.draws(ref.rng_task_key(100, 1, call_no, 0, fid), 20, n)[0]
    fr = Frames(w, rows=[0], counts=[n])
    pa, pb = fr.pa.reshape(-1, 2), fr.pb.reshape(-1, 2)
    pa[b], pb[b] = pa[a], pb[a]
    fr.pa, fr.pb = pa.reshape(-1).copy(), pb.reshape(-1).copy()
    return fr, (a, b)


@needs2
def test_panic_on_a_replica_share_gives_the_single_device_message(rsb, synth_mod):
    w = workload("small")
    n, G, c_star = w.n_rays, N_GPUS, 977
    fr, pair = _panic_frame(w, c_star, n)
    D = rsb.presync_delays(0.0, 0.005, 0.02).size
    m = 2 * G  # the primary takes readouts 0 and 1, the last device the last two
    # call numbers none of whose draws (at any delay) is the equal pair: their grids are finite
    clean = (c for c in itertools.count() if c != c_star and all(
        {x, y} != set(pair) for d in range(D) for x, y in ref.draws(ref.rng_task_key(100, 1, c, d, fr.fb), 20, n)))
    calls = np.array(list(itertools.islice(clean, m)), dtype=np.uint64)
    one, many = _pair(rsb, w)
    for p in (one, many):
        fr.ingest(p, synth_mod, synth_mod.READOUT)
    readouts = np.linspace(0.0, 0.02, m)
    args = (readouts, 0.0, fr.fb, fr.fe, 0.005, 0.02)
    c1, _ = one.readout_search(*args, call_nos=calls)
    c2, _ = many.readout_search(*args, call_nos=calls)
    assert np.array_equal(c1, c2) and np.isfinite(c1).all()
    for where in ([m - 1], [G, m - 1], [2, m - 2]):  # shares of the devices after the primary
        bad = calls.copy()
        bad[where] = c_star
        a, b = _error(rsb, one, *args, call_nos=bad), _error(rsb, many, *args, call_nos=bad)
        assert a == b == (rsb.E_NONFINITE, "pre-sync: non-finite r", 0)


@needs2
def test_multi_device_traffic(rsb, synth_mod):
    w = workload("small")
    fr = Frames(w)
    one, many = _pair(rsb, w)
    for p in (one, many):
        fr.ingest(p, synth_mod, synth_mod.READOUT)
    table = many.frame_table()
    arena = int(max(int(f["off"]) + (int(f["n"]) + 31) // 32 * 32 for f in table))
    nq = many.stats()["gyro_samples"]
    delays = rsb.presync_delays(INITIAL, STEP, RADIUS)

    def delta(fn):
        s0 = many.stats()
        out = fn()
        s1 = many.stats()
        return out, s1["broadcast_bytes"] - s0["broadcast_bytes"], s1["nccl_calls"] - s0["nccl_calls"]

    for p in (one, many):
        p.set_rng(100, 1)
    # as the parent commit: the first compute call replicates the spline records and the arena (one piece:
    # the pixels ingest leaves no chunk in flight) and gathers once; a grid call after it only gathers
    out, nb, nc = delta(lambda: many.PreSync(INITIAL, fr.fb, fr.fe, STEP, RADIUS))
    assert out == one.PreSync(INITIAL, fr.fb, fr.fe, STEP, RADIUS)
    assert (nb, nc) == (nq * 128 + arena * 72, 3)
    out, nb, nc = delta(lambda: many.presync_grid(fr.fb, fr.fe, delays, call_no=4))
    assert np.array_equal(out, one.presync_grid(fr.fb, fr.fe, delays, call_no=4)) and (nb, nc) == (0, 1)
    # the first search sends the plane, a second one nothing
    out, nb, nc = delta(lambda: _search(many, fr.fb, fr.fe))
    _equal(out, _search(one, fr.fb, fr.fe))
    assert (nb, nc) == (16 * arena, 1)
    out, nb, nc = delta(lambda: _search(many, fr.fb, fr.fe, call_nos=[9] * len(READOUTS)))
    _equal(out, _search(one, fr.fb, fr.fe, call_nos=[9] * len(READOUTS)))
    assert (nb, nc) == (0, 0)
    # a PreSync after the searches: as before them
    out, nb, nc = delta(lambda: many.presync_grid(fr.fb, fr.fe, delays, call_no=5))
    assert np.array_equal(out, one.presync_grid(fr.fb, fr.fe, delays, call_no=5)) and (nb, nc) == (0, 1)

    def resend_after(change):
        for p in (one, many):
            change(p)
        many.presync_grid(fr.fb, fr.fe, delays, call_no=6)  # replicates the arena, not the plane
        rays = many.device_state()["arena_rays"]
        out, nb, nc = delta(lambda: _search(many, fr.fb, fr.fe))
        _equal(out, _search(one, fr.fb, fr.fe))
        assert (nb, nc) == (16 * rays, 1)

    w2 = workload("small", seed=9)
    R2 = 0.0141
    # a new pixels ingest (in place)
    resend_after(lambda p: Frames(w2).ingest(p, synth_mod, R2))
    # a new pixels frame outside the searched range (it grows the arena), then a rays overwrite of it
    extra = fr.fe + 10
    resend_after(lambda p: Frames(w2, rows=[3], ids=[extra]).ingest(p, synth_mod, R2))
    resend_after(lambda p: p.set_track_batch(np.array([extra]), np.array([w.n_rays], dtype=np.uint64), w.ts_a[3],
                                             w.ts_b[3], w.rays_a[3].reshape(-1), w.rays_b[3].reshape(-1)))
    # arena growth: frames appended by a rays form beyond the arena's capacity
    ids = fr.fe + 1000 + np.arange(w.n_frames)
    resend_after(lambda p: p.set_track_batch(ids, np.full(w.n_frames, w.n_rays, dtype=np.uint64), w.ts_a.reshape(-1),
                                             w.ts_b.reshape(-1), w.rays_a.reshape(-1), w.rays_b.reshape(-1)))


@needs2
def test_set_readout_on_a_multi_device_problem(rsb, synth_mod):
    w = workload("small")
    fr = Frames(w)
    one, many = _pair(rsb, w)
    fr.ingest(many, synth_mod, synth_mod.READOUT)
    many.set_rng(100, 1)
    _search(many, fr.fb, fr.fe)  # the replicas hold the row fractions
    R2 = 0.0163
    many.set_readout(R2, fr.fb, fr.fe)
    fr.ingest(one, synth_mod, R2)
    delays = rsb.presync_delays(INITIAL, STEP, RADIUS)
    for p in (one, many):
        p.set_rng(100, 3)
    assert many.PreSync(INITIAL, fr.fb, fr.fe, STEP, RADIUS) == one.PreSync(INITIAL, fr.fb, fr.fe, STEP, RADIUS)
    assert np.array_equal(many.presync_grid(fr.fb, fr.fe, delays, call_no=8), one.presync_grid(fr.fb, fr.fe, delays,
                                                                                                call_no=8))
    # and a search after it: the arena went out again, the row fractions did not need to
    _equal(_search(many, fr.fb, fr.fe), _search(one, fr.fb, fr.fe))


# ---- 3. one process per GPU (sharded.py over NCCL) -----------------------------------------------------
def _nccl_worker(rank, world, port, q, readouts):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    rsb = importlib.import_module("rs-sync_b200")
    synth_mod = importlib.import_module("rs-sync_b200.synth")
    sh = _sharded()
    w = workload("small")
    half = w.n_frames // 2
    pix, rows = Frames(w, rows=range(half)), Rows(w, synth_mod, rows=range(half, w.n_frames))
    if rank == 0:
        p = _problem(rsb, w)
        pix.ingest(p, synth_mod, synth_mod.READOUT)
        rows.ingest(p, synth_mod.READOUT)
    else:
        p = rsb.SyncProblem(seed=100)
    dev = f"cuda:{rank}"
    sh.replicate_state(p, rank=rank, world=world, device=dev)
    sh.replicate_row_fractions(p, rank=rank, world=world, device=dev)
    out = sh.readout_search_sharded(p, readouts, INITIAL, pix.fb, rows.fe, STEP, RADIUS, call_no_base=5, rank=rank,
                                    world=world, device=dev, curves=True)
    q.put((rank, [np.asarray(x) for x in out]))
    dist.barrier()
    dist.destroy_process_group()


@needs2
def test_sharded_over_nccl_ranks(rsb, synth_mod):
    import torch.multiprocessing as mp
    readouts = np.linspace(-0.004, 0.024, 7)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() + 1313) % 2000
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q, readouts)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=300) for _ in range(2))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    w = workload("small")
    half = w.n_frames // 2
    pix, rows = Frames(w, rows=range(half)), Rows(w, synth_mod, rows=range(half, w.n_frames))
    one = _problem(rsb, w)
    pix.ingest(one, synth_mod, synth_mod.READOUT)
    rows.ingest(one, synth_mod.READOUT)
    want = one.readout_search(readouts, INITIAL, pix.fb, rows.fe, STEP, RADIUS, call_nos=5 + np.arange(7), curves=True)
    for rank in range(2):
        assert all(np.array_equal(x, y) for x, y in zip(got[rank], want))
