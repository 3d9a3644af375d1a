"""The frames of tests/estimator_frames.py on the CPU oracle: every builder's preconditions hold, the
oracle's estimator returns the winner of its own per-hypothesis trace, and (where oracle/_ref is built)
the compiled reference breaks the designed ties the same way as the strict oracle."""
import numpy as np
import pytest

import estimator_frames as ef
from conftest import workload

# (t1, t2, iters): the first hypothesis (no best yet), the two halves of one packed pair (t even), two
# adjacent pairs (t odd), the last of 20; for 200, across the 32-hypothesis batch boundary and inside
# the last partial batch.  Five rays have 20 ordered row pairs: long before hypothesis 31 one repeats.
TIES = [(0, 1, 20), (2, 3, 20), (5, 6, 20), (7, 19, 20), (31, 32, 200), (193, 198, 200)]


def tie_cases(n):
    return [c for c in TIES if n >= 32 or c[2] == 20]


def stream_of(iters):
    return ef.STREAM_PRESYNC if iters == 20 else ef.STREAM_SYNCINIT


def assert_oracle_is_trace(oracle_loader, f):
    o = ef.oracle_problem(oracle_loader, [f])
    v, q, best = o.estimator_trace(f.fid, 0.0, f.iters, f.stream, f.call_no, f.offset)
    m, _ = o.guess_motion(f.fid, 0.0, f.iters, f.stream, f.call_no, f.offset)
    assert np.array_equal(ef.bits(m), ef.bits(v[best]))
    assert np.all(q[:best] > q[best]) and np.all(q[best:] >= q[best])
    return v, q, best


@pytest.mark.parametrize("n", ef.N_RAYS)
def test_mirror_frames(oracle_loader, n):
    for t1, t2, iters in tie_cases(n):
        f = ef.mirror_frame(n, t1, t2, iters, stream_of(iters), oracle_loader=oracle_loader)
        ef.check_mirror(f, oracle_loader)
        _, _, best = assert_oracle_is_trace(oracle_loader, f)
        assert best == t1
        # the rows of the tied pair are mirror images of each other, bit for bit
        P = ef.oracle_problem(oracle_loader, [f]).problem_matrix(f.fid, 0.0, n)
        d = ef._draws(f.fid, n, f.stream, f.call_no, f.offset, iters)
        for i, j in zip(d[t1], d[t2]):
            assert np.array_equal(ef.bits(P[j]), ef.bits(P[i] * [1.0, -1.0, -1.0]))


@pytest.mark.parametrize("n", [n for n in ef.N_RAYS if n >= 32])
def test_near_tie_sweeps(oracle_loader, n):
    """the builder's preconditions (asserted inside) and the oracle's winner on every frame"""
    for iters in (20, 200):
        frames = ef.near_tie_sweep(n, iters, stream_of(iters), oracle_loader=oracle_loader)
        assert len({f.fid for f in frames}) == 1  # one frame id, the rays of t2 rotated in place
        for f in frames:
            _, _, best = assert_oracle_is_trace(oracle_loader, f)
            assert best == f.meta["best"]


@pytest.mark.parametrize("zero_vector", [False, True], ids=["mixed", "zero-vector"])
@pytest.mark.parametrize("n", ef.N_RAYS)
def test_zero_quartile_frames(oracle_loader, n, zero_vector):
    for iters in (20, 200):
        f = ef.zero_frame(n, zero_vector, t1=0 if n < 64 else 3, iters=iters, stream=stream_of(iters),
                          oracle_loader=oracle_loader)
        ef.check_zero(f, oracle_loader)
        _, q, best = assert_oracle_is_trace(oracle_loader, f)
        assert best == f.t1
        # the tie is not a one-off: quartile 0 at other keys (other delays of a grid) too
        o = ef.oracle_problem(oracle_loader, [f])
        zeros = [o.estimator_trace(f.fid, 0.0, iters, f.stream, f.call_no, off)[1].min() == 0.0 for off in range(8)]
        assert all(zeros)


@pytest.mark.parametrize("n", ef.N_RAYS)
def test_repeated_pair_frames(oracle_loader, n):
    for iters in (20, 200):
        f = ef.repeated_frame(n, iters, stream_of(iters))
        P = ef.oracle_problem(oracle_loader, [f]).problem_matrix(f.fid, 0.0, n)
        g = f.meta["group"]
        for k in np.unique(g):  # copies of one ray pair have bit-identical rows, so equal residual keys
            rows = ef.bits(P[g == k])
            assert len(rows) >= 2 and (rows == rows[0]).all()
        _, q, best = assert_oracle_is_trace(oracle_loader, f)
        d = ef._draws(f.fid, n, f.stream, f.call_no, f.offset, iters)
        if all(g[a] != g[b] for a, b in d):
            assert q[best] > 0.0  # the winner's quartile is a real residual key, not the zero hypothesis


def threshold_cases(n):
    """(iters, stream) for which threshold_rows_frame finds a frame of n rays"""
    return [(20, ef.STREAM_PRESYNC)] * (n >= 32) + [(200, ef.STREAM_SYNCINIT)] * (n >= 225)


@pytest.mark.parametrize("n", [n for n in ef.N_RAYS if n >= 32])
def test_threshold_row_frames(oracle_loader, n):
    """rows of norm just below 1e-12: left unscaled (the oracle's winner is its trace's), and whether
    they are decides the winner (asserted by the builder)"""
    for iters, stream in threshold_cases(n):
        f = ef.threshold_rows_frame(n, iters, stream, oracle_loader=oracle_loader)
        P = ef.oracle_problem(oracle_loader, [f]).problem_matrix(f.fid, 0.0, n)
        nrm = np.linalg.norm(P[f.meta["rows"]], axis=1)
        assert np.all(nrm < 1e-12) and np.all(np.float32(nrm * nrm) == np.float32(1e-24))
        _, _, best = assert_oracle_is_trace(oracle_loader, f)
        assert best == f.t1 != f.t2


def static_problem(oracle_loader, w, frames):
    o = oracle_loader.OracleProblem(threads=2, seed=ef.SEED).load(w)
    for f in frames:
        f.load(o)
    return o


@pytest.mark.parametrize("drawn", [False, True], ids=["avoided", "drawn"])
def test_static_pair_frames(oracle_loader, drawn):
    w = workload("tiny", first_frame=200)
    for i, k in ((2, 0), (7, 5)):
        f = ef.with_static_pair(w, i, k, drawn=drawn)
        o = static_problem(oracle_loader, w, [f])
        s = f.meta["static"]
        for delay in (0.0, 0.03):
            P = o.problem_matrix(f.fid, delay, w.n_rays)
            assert np.all(np.isfinite(P))
            assert np.linalg.norm(P[s]) < 1e-12 and np.min(np.linalg.norm(np.delete(P, s, 0), axis=1)) > 1e-9
        v, q, best = o.estimator_trace(f.fid, 0.0, 20, f.stream, f.call_no, f.offset)
        d = ef._draws(f.fid, w.n_rays, f.stream, f.call_no, f.offset, 20)
        assert (s in {x for ab in d for x in ab}) == drawn
        if drawn:  # the tiny hypothesis (left unnormalised, |v| ~ |row|) wins
            assert s in d[best] and np.linalg.norm(v[best]) < 1e-12
        _, c_flags = _presync_flags(o, f.fid)
        assert c_flags == 0


def _presync_flags(o, fid):
    c, _, flags = o.presync_grid(fid, fid + 1, np.linspace(-0.04, 0.04, 9), frame_costs=True)
    return c, flags


def test_all_static_frame_flags(oracle_loader):
    """every row tiny but finite: whatever else the frame does, it does not raise pre_sync's P flag"""
    w = workload("tiny", first_frame=200)
    f = ef.all_static(w, 0)
    o = static_problem(oracle_loader, w, [f])
    P = o.problem_matrix(f.fid, 0.0, w.n_rays)
    assert np.all(np.isfinite(P)) and np.max(np.linalg.norm(P, axis=1)) < 1e-12
    _, flags = _presync_flags(o, f.fid)
    assert flags & 1 == 0


ref_loader = pytest.importorskip("oracle.ref_loader")
needs_ref = pytest.mark.skipif(not ref_loader.available(), reason="oracle/_ref not built")


@needs_ref
@pytest.mark.parametrize("n", [5, 33, 257])
def test_reference_breaks_ties_like_the_oracle(oracle_loader, n):
    """the strict oracle (the reference's own expression order) and the compiled reference pick the
    same hypothesis of an exact tie, the earlier one: M of t1, not the mirrored M of t2"""
    frames = [ef.mirror_frame(n, t1, t2, iters, stream_of(iters), oracle_loader=oracle_loader)
              for t1, t2, iters in tie_cases(n)]
    frames += [ef.zero_frame(n, zv, oracle_loader=oracle_loader) for zv in (False, True)]
    for f in frames:
        v, q, best = f.trace(oracle_loader)
        o = ef.oracle_problem(oracle_loader, [f])
        o.set_strict(True)
        r = ef.load_gyro(ref_loader.RefProblem(threads=2, seed=ef.SEED))
        f.load(r)
        mo, _ = o.guess_motion(f.fid, 0.0, f.iters, f.stream, f.call_no, f.offset)
        mr = r.guess_motion(f.fid, 0.0, f.iters, f.stream, f.call_no, f.offset)
        assert np.array_equal(mo, mr), (f.family, n, mo, mr)
        assert np.max(np.abs(mr - v[f.t1])) <= 1e-12 < np.max(np.abs(mr - v[f.t2])), (f.family, n)
