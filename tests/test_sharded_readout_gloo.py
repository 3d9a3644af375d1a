"""world_size-2 gloo test of sharded.readout_search_sharded on CPU, with a fake problem whose results are a
function of (readout, call number): what is under test is the round-robin of the readouts over the ranks,
the call numbers each rank passes, the gather and the order of the gathered (cost, delay, curve) rows."""
import importlib
import os
import sys

import numpy as np
import torch.multiprocessing as mp

from conftest import ROOT

D = 3
BASE = 40
SIZES = (0, 1, 2, 3, 11)


class FakeProblem:
    """readout_search as the engine's wrapper shapes it; records what it was asked"""

    def __init__(self):
        self.asked = []

    def readout_search(self, readouts, initial_delay, frame_begin, frame_end, search_step, search_radius,
                       call_nos=None, curves=False):
        r = np.asarray(readouts, dtype=np.float64)
        c = np.asarray(call_nos, dtype=np.uint64)
        self.asked.append((r.tolist(), c.tolist(), (initial_delay, frame_begin, frame_end, search_step,
                                                    search_radius), curves))
        costs, delays = expected(r, c)
        if curves:
            return costs, delays, expected_curves(r, c)
        return costs, delays


def expected(r, c):
    c = np.asarray(c, dtype=np.float64)
    return 1000.0 * r + c, 0.5 * c - r


def expected_curves(r, c):
    return np.asarray(r)[:, None] * 10.0 + np.asarray(c, dtype=np.float64)[:, None] + np.arange(D)[None, :] * 0.25


def _readouts(n):
    return 0.001 * np.arange(n) + 0.0123


def _worker(rank, world, port, q):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sharded = importlib.import_module("rs-sync_b200.sharded")
    out = {}
    for n in SIZES:
        for curves in (False, True):
            fake = FakeProblem()
            res = sharded.readout_search_sharded(fake, _readouts(n), 0.01, 7, 19, 0.002, 0.1, call_no_base=BASE,
                                                 rank=rank, world=world, curves=curves)
            out[(n, curves)] = ([np.asarray(x) for x in res], fake.asked)
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


def test_readouts_round_robin_world2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() + 977) % 2000
    world = 2
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for n in SIZES:
        r = _readouts(n)
        calls = BASE + np.arange(n)
        want_c, want_d = expected(r, calls)
        for curves in (False, True):
            for rank in range(world):
                res, asked = got[rank][(n, curves)]
                # one call per rank, even without readouts, with readouts rank, rank + world, ... and their
                # call numbers
                assert len(asked) == 1
                ar, ac, args, acurves = asked[0]
                assert ar == r[rank::world].tolist() and ac == calls[rank::world].tolist()
                assert args == (0.01, 7, 19, 0.002, 0.1) and acurves == curves
                # every rank holds every result, in readout order
                assert len(res) == (3 if curves else 2)
                assert np.array_equal(res[0], want_c) and np.array_equal(res[1], want_d)
                if curves:
                    assert res[2].shape == (n, D)
                    assert np.array_equal(res[2], expected_curves(r, calls))


def test_one_rank_is_the_problem_itself():
    sharded = importlib.import_module("rs-sync_b200.sharded")
    fake = FakeProblem()
    r = _readouts(5)
    c, d, cv = sharded.readout_search_sharded(fake, r, 0.0, 0, 10, 0.002, 0.1, call_no_base=3, curves=True)
    assert fake.asked[0][1] == [3, 4, 5, 6, 7]
    want_c, want_d = expected(r, 3 + np.arange(5))
    assert np.array_equal(c, want_c) and np.array_equal(d, want_d)
    assert np.array_equal(cv, expected_curves(r, 3 + np.arange(5)))
