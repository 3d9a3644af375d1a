"""Frames built so that the translation estimator (opt_guess_translational_motion, core_private.cpp:34-59)
must break ties, settle near ties and select among equal keys, for tests/test_estimator_ties.py and
tests/test_gpu_estimator_ties.py.

Random synthetic frames practically never tie: two different hypotheses with exactly the same quartile
need structure.  Families a-d use a constant gyro track (1, 0, 0, 0): its spline is exactly the identity
and de-rotation returns a ray bit for bit, so a frame's rows are the contract's cross products of its
rays, the same at every delay.  The draws of a task (which caller indices each hypothesis comes from)
are known in advance from its RNG key (plain_reference.draws), so a builder places the rays a tie needs
where the draws will pick them.  Every builder checks its own preconditions on the oracle's trace of
the estimator (OracleProblem.estimator_trace) and, where a scene seed or frame id does not meet them,
tries the next one in a fixed order: the frames are the same on every run.

Families:
  a  mirror frames: hypotheses t1 < t2 tie exactly with different M;
  b  family a with t2's rays rotated by eps: the quartile gap sweeps across the fp32 band;
  c  zero quartiles: rows (0, c, 0) give many hypotheses quartile exactly 0;
  d  repeated ray pairs: equal residual keys at the quartile rank;
  e  a static ray pair (a feature that does not move under no rotation): a finite row of norm < 1e-12.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

import plain_reference as pr

SEED = 100                  # the problems' RNG seed
STREAM_PRESYNC, STREAM_SYNCINIT = 1, 3
K_MARGIN = 1.4e-6           # the fp32 tournament's margin (engine.cu, kMargin)
GYRO_RATE, GYRO_T0, GYRO_N = 200.0, 0.0, 400
FPS = 30.0
QUATS = np.tile(np.array([1.0, 0.0, 0.0, 0.0]), (GYRO_N, 1))
N_RAYS = [5, 32, 33, 64, 65, 129, 225, 257, 385, 512]  # every SLOTS instantiation, every n mod 4


@dataclass
class Frame:
    """one frame and the task it was designed for: (stream, call_no, offset_idx, iters) at any delay"""
    family: str
    fid: int
    ts_a: np.ndarray
    ts_b: np.ndarray
    rays_a: np.ndarray
    rays_b: np.ndarray
    stream: int
    call_no: int
    offset: int
    iters: int
    t1: int = -1            # the hypothesis that must win
    t2: int = -1            # one that ties (a, c) or nearly ties (b) with it
    meta: dict = field(default_factory=dict)

    @property
    def n(self):
        return int(self.ts_a.shape[0])

    def key(self):
        return pr.rng_task_key(SEED, self.stream, self.call_no, self.offset, self.fid)

    def load(self, p):
        p.SetTrackResult(self.fid, self.ts_a, self.ts_b, self.rays_a, self.rays_b, self.n)
        return p

    def trace(self, oracle_loader, delay=0.0):
        return oracle_problem(oracle_loader, [self]).estimator_trace(self.fid, delay, self.iters, self.stream,
                                                                     self.call_no, self.offset)


def load_gyro(p):
    p.SetGyroQuaternions(QUATS, GYRO_N, GYRO_RATE, GYRO_T0)
    return p


def oracle_problem(oracle_loader, frames, threads=2):
    o = load_gyro(oracle_loader.OracleProblem(threads=threads, seed=SEED))
    for f in frames:
        f.load(o)
    return o


def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def _timestamps(fid, n):
    ts_a = fid / FPS + np.linspace(0.0, 0.02, n)
    return ts_a, ts_a + 1.0 / FPS


def _draws(fid, n, stream, call_no, offset, iters):
    return pr.draws(pr.rng_task_key(SEED, stream, call_no, offset, fid), iters, n)


def _scene_pair(rng, T, noise, outlier):
    """a ray pair viewing a static point from the origin and from T (noise: radians on b)"""
    X = np.array([rng.uniform(-1.5, 1.5), rng.uniform(-1.0, 1.0), rng.uniform(2.0, 6.0)])
    a = _unit(X)
    b = _unit(X - T) if not outlier else _unit(np.array([rng.uniform(-0.5, 0.5), rng.uniform(-0.5, 0.5), 1.0]))
    if noise:
        b = _unit(b + rng.normal(0.0, noise, 3))
    return a, b


def bits(v):
    return np.ascontiguousarray(v, dtype=np.float64).view(np.uint64)


def sqrt_gap(q, s, t):
    """|sqrt(q_s) - sqrt(q_t)|: the fp32 tournament's margin is a distance in this domain"""
    return abs(float(np.sqrt(q[s])) - float(np.sqrt(q[t])))


# ---- a: exact ties --------------------------------------------------------------------------------
def _mirror(v):
    return v * np.array([-1.0, 1.0, 1.0])


def mirror_frame(n, t1, t2, iters=20, stream=STREAM_PRESYNC, call_no=0, offset=0, fid0=1000,
                 oracle_loader=None, eps=0.0):
    """Rays in x-mirror pairs (x, y, z) <-> (-x, y, z) under an involution sigma on caller indices, with
    sigma(a1) = a2 and sigma(b1) = b2 for the draws (a1, b1) of t1 and (a2, b2) of t2.  Every operation of
    the contract is sign-symmetric under the mirror, so the rows of i and sigma(i) are (r0, r1, r2) and
    (r0, -r1, -r2), t2's hypothesis is (vx, -vy, -vz) and its multiset of residuals is t1's: the two
    quartiles are equal in binary64.  Rays a1, b1 (and their images) are noise-free views of static
    points under a translation (0, ty, tz); the others carry noise and outliers, so the tied pair wins.
    eps != 0 (family b): the ray pairs a2 and b2 are then rotated by eps about the x axis."""
    assert t1 < t2 < iters
    fid = fid0
    for attempt in range(4000):
        fid = fid0 + attempt
        d = _draws(fid, n, stream, call_no, offset, iters)
        (a1, b1), (a2, b2) = d[t1], d[t2]
        if len({a1, b1, a2, b2}) < 4:
            continue
        rng = np.random.default_rng([fid, n, t1, t2])
        T = np.array([0.0, rng.uniform(-0.3, 0.3), rng.uniform(0.5, 1.0)])
        sigma = {a1: a2, a2: a1, b1: b2, b2: b1}
        rest = [i for i in rng.permutation(n) if i not in sigma]
        fixed = rest.pop() if len(rest) % 2 else None
        for i, j in zip(rest[0::2], rest[1::2]):
            sigma[int(i)], sigma[int(j)] = int(j), int(i)
        ra, rb = np.empty((n, 3)), np.empty((n, 3))
        done = set()
        for i in range(n):
            if i in done or i == fixed:
                continue
            clean = i in (a1, b1, a2, b2)
            a, b = _scene_pair(rng, T, 0.0 if clean else 2e-3, (not clean) and rng.uniform() < 0.25)
            ra[i], rb[i] = a, b
            ra[sigma[i]], rb[sigma[i]] = _mirror(a), _mirror(b)
            done |= {i, sigma[i]}
        if fixed is not None:  # its own mirror image: a pair in the plane x = 0
            a, b = _scene_pair(rng, T, 2e-3, False)
            ra[fixed], rb[fixed] = a * [0.0, 1.0, 1.0], b * [0.0, 1.0, 1.0]
        if eps:
            c, s = np.cos(eps), np.sin(eps)
            R = np.array([[1.0, 0.0, 0.0], [0.0, c, -s], [0.0, s, c]])
            for i in (a2, b2):
                ra[i], rb[i] = R @ ra[i], R @ rb[i]
        ts_a, ts_b = _timestamps(fid, n)
        f = Frame("b" if eps else "a", fid, ts_a, ts_b, ra, rb, stream, call_no, offset, iters, t1, t2,
                  meta=dict(eps=eps))
        if eps or oracle_loader is None:
            return f
        v, q, best = f.trace(oracle_loader)
        if q[t1] == q[t2] and best == t1:
            check_mirror(f, oracle_loader)
            return f
    raise AssertionError(f"no mirror frame for n={n}, ties {t1}, {t2}")


def check_mirror(f, oracle_loader):
    """family a's preconditions: the tie is exact, the tied M differ in bits, t1 is the first strict
    minimum (t2 is then not strictly below it either)"""
    v, q, best = f.trace(oracle_loader)
    assert q[f.t1] == q[f.t2], (f.n, f.t1, f.t2, q[f.t1], q[f.t2])
    assert not np.array_equal(bits(v[f.t1]), bits(v[f.t2]))
    assert np.array_equal(bits(v[f.t2]), bits(v[f.t1] * [1.0, -1.0, -1.0]))
    assert best == f.t1 and np.all(q[:f.t1] > q[f.t1])
    return v, q, best


# ---- b: near ties across the fp32 margin ---------------------------------------------------------
EPS_GRID = [s * e for e in 10.0 ** np.arange(-12.0, -2.4, 0.75) for s in (1.0, -1.0)]


def near_tie_sweep(n, iters=20, stream=STREAM_PRESYNC, call_no=0, offset=0, oracle_loader=None):
    """family a with t1 = 0 (the tournament's first best, so that t2 is compared with t1 and nothing
    else decides the settle) and the rays of t2 rotated by each eps of EPS_GRID.  Returns the frames
    (one id per eps) with meta['gap'] = sqrt-domain quartile gap of t2 against t1 from the trace.
    Preconditions: the winner is t1 or t2 at every eps, every other hypothesis is more than
    2 kMargin from both in the sqrt domain, the gap runs from below 0.05 kMargin to above 2 kMargin,
    and t2 is better than t1 at some eps and worse at others."""
    t1, t2 = 0, iters - 1
    for attempt in range(40):
        base = mirror_frame(n, t1, t2, iters, stream, call_no, offset, fid0=5000 + 97 * attempt,
                            oracle_loader=oracle_loader)
        frames, ok = [], True
        for k, eps in enumerate(EPS_GRID):
            f = mirror_frame(n, t1, t2, iters, stream, call_no, offset, fid0=base.fid, eps=eps)
            v, q, best = f.trace(oracle_loader)
            others = [t for t in range(iters) if t not in (t1, t2)]
            if best not in (t1, t2) or min(min(sqrt_gap(q, t, t1), sqrt_gap(q, t, t2)) for t in others) <= 2 * K_MARGIN:
                ok = False
                break
            f.meta.update(gap=sqrt_gap(q, t1, t2), t2_better=bool(q[t2] < q[t1]), best=best)
            frames.append(f)
        if not ok:
            continue
        gaps = [f.meta["gap"] for f in frames]
        better = [f.meta["t2_better"] for f in frames]
        if min(gaps) < 0.05 * K_MARGIN and max(gaps) > 2 * K_MARGIN and any(better) and not all(better):
            return frames
    raise AssertionError(f"no near-tie sweep for n={n}")


# ---- c: zero quartiles ---------------------------------------------------------------------------
def zero_frame(n, zero_vector, t1=0, iters=20, stream=STREAM_PRESYNC, call_no=0, offset=0, fid0=20000,
               oracle_loader=None):
    """Rays with y = 0 exactly give rows (0, c, 0) (signed zeros aside); a hypothesis built from one has
    v_y = 0 exactly and so residual exactly 0 on all of them.  n/4 + 1 or more such rows give every such
    hypothesis quartile 0: ties between different M in every task and at every delay.  A hypothesis
    from two of them is the zero vector (the reference's "non-finite r").  Hypothesis t1 is the first
    to draw one: with one of its rows among them (zero_vector=False) or both (True)."""
    m = n // 4 + 1 + n // 8
    for attempt in range(4000):
        fid = fid0 + attempt
        d = _draws(fid, n, stream, call_no, offset, iters)
        early = {i for ab in d[:t1] for i in ab}
        a1, b1 = d[t1]
        if a1 in early or b1 in early:
            continue
        Z = [a1, b1] if zero_vector else [a1]
        pool = [i for i in range(n) if i not in early and i not in (a1, b1)]
        rng = np.random.default_rng([fid, n, 3])
        if len(pool) < m - len(Z):
            continue
        Z += [int(i) for i in rng.choice(pool, m - len(Z), replace=False)]
        T = _unit(np.array([rng.uniform(-0.5, 0.5), rng.uniform(-0.5, 0.5), 1.0]))
        ra, rb = np.empty((n, 3)), np.empty((n, 3))
        for i in range(n):
            ra[i], rb[i] = _scene_pair(rng, T, 2e-3, rng.uniform() < 0.2)
        for i in Z:
            ra[i, 1] = rb[i, 1] = 0.0
        ts_a, ts_b = _timestamps(fid, n)
        f = Frame("c0" if zero_vector else "c", fid, ts_a, ts_b, ra, rb, stream, call_no, offset, iters, t1,
                  meta=dict(zeros=sorted(Z)))
        v, q, best = f.trace(oracle_loader)
        later = [t for t in range(t1 + 1, iters) if q[t] == 0.0 and not np.array_equal(bits(v[t]), bits(v[t1]))]
        if later:
            f.t2 = later[0]
            check_zero(f, oracle_loader)
            return f
    raise AssertionError(f"no zero-quartile frame for n={n}")


def check_zero(f, oracle_loader):
    v, q, best = f.trace(oracle_loader)
    assert best == f.t1 and q[f.t1] == 0.0 and q[f.t2] == 0.0
    assert np.all(q[:f.t1] > 0.0)
    assert not np.array_equal(bits(v[f.t1]), bits(v[f.t2]))
    assert (not np.any(v[f.t1])) == (f.family == "c0")
    return v, q, best


# ---- d: equal keys at rank n/4 -------------------------------------------------------------------
def repeated_frame(n, iters=20, stream=STREAM_PRESYNC, call_no=0, offset=0, fid0=30000, rep=3):
    """Every ray pair (a != b) repeated rep times at scattered caller indices: identical rows have
    bit-identical residuals, so every key (the one at rank n/4 among them) is one of rep equal keys.
    Two copies of one row drawn together make the zero hypothesis, which would win with quartile 0;
    where the draws can avoid that (at least 1 % of keys do) the designed task's draws never do."""
    groups = -(-n // rep)
    avoid = (1.0 - (rep - 1) / (n - 1)) ** iters > 0.01
    for attempt in range(4000):
        fid = fid0 + attempt
        rng = np.random.default_rng([fid, n, 4])
        src = rng.permutation(np.arange(n) % groups)  # caller index -> its group
        d = _draws(fid, n, stream, call_no, offset, iters)
        if avoid and any(src[a] == src[b] for a, b in d):
            continue
        T = _unit(np.array([rng.uniform(-0.5, 0.5), rng.uniform(-0.5, 0.5), 1.0]))
        pairs = [_scene_pair(rng, T, 2e-3, rng.uniform() < 0.2) for _ in range(groups)]
        ra = np.array([pairs[g][0] for g in src])
        rb = np.array([pairs[g][1] for g in src])
        ts_a, ts_b = _timestamps(fid, n)
        return Frame("d", fid, ts_a, ts_b, ra, rb, stream, call_no, offset, iters, meta=dict(group=src))
    raise AssertionError(f"no repeated-pair frame for n={n}")


# ---- e: tiny finite rows -------------------------------------------------------------------------
def with_static_pair(w, i, k, stream=STREAM_PRESYNC, call_no=0, offset=0, iters=20, drawn=None):
    """Frame i of a synth workload (random gyro) with ray pair k made static: b = a and ts_b = ts_a.
    Both rays are de-rotated by the same quaternion, so the row is the rounding residue of a cross
    product (|row| < 1e-12, finite).  drawn=False / True: the static pair is instead the k-th (cyclically)
    of the ray pairs that the designed task's draws avoid / include (None: pair k itself)."""
    n = w.n_rays
    fid = int(w.frame_ids[i])
    d = _draws(fid, n, stream, call_no, offset, iters)
    hit = {x for ab in d for x in ab}
    if drawn is not None:
        cand = [j for j in range(n) if (j in hit) == drawn]
        assert cand, (fid, drawn)
        k = cand[k % len(cand)]
    ts_a, ts_b = w.ts_a[i].copy(), w.ts_b[i].copy()
    ra, rb = w.rays_a[i].copy(), w.rays_b[i].copy()
    rb[k], ts_b[k] = ra[k], ts_a[k]
    return Frame("e", fid, ts_a, ts_b, ra, rb, stream, call_no, offset, iters, meta=dict(static=k))


def all_static(w, i):
    """the frame of test_estimator_degenerate_scenes: one ray, n times, a = b, ts_b = ts_a"""
    n = w.n_rays
    same = np.tile(w.rays_a[i][:1], (n, 1))
    return Frame("e0", 10 ** 4, w.ts_a[i].copy(), w.ts_a[i].copy(), same, same.copy(), STREAM_PRESYNC, 0, 0, 20)


# ---- e': rows at the normalisation threshold -----------------------------------------------------
S_BELOW = 1e-12 * (1.0 - 1e-8)  # safe_normalize leaves a row of this norm unscaled; fp32(|row|^2) == fp32(1e-24)


def threshold_rows_frame(n, iters=20, stream=STREAM_PRESYNC, call_no=0, offset=0, fid0=90000, oracle_loader=None):
    """A noisy frame with n/8 (at least 1) ray pairs whose rows are S_BELOW times a unit axis, exactly:
    (0, 0, 1) x (s, 0, 1) = (0, s, 0) and the like.  safe_normalize leaves them unscaled, so under the
    contract their residuals are ~1e-24 for every hypothesis; a row normalised to unit length would
    instead have residual v_y^2.  The frame is kept where that difference moves the winner by more
    than 4 kMargin in the sqrt domain: an estimator that normalised these rows would certify the wrong
    hypothesis.  The designed task's draws avoid those rows (a hypothesis through one of them would be
    ~1e-12 long, left unnormalised, and win)."""
    k = max(1, n // 8)
    axes = [(np.array([0.0, 0.0, 1.0]), np.array([S_BELOW, 0.0, 1.0])),
            (np.array([0.0, 1.0, 0.0]), np.array([S_BELOW, 1.0, 0.0])),
            (np.array([0.0, 0.0, 1.0]), np.array([0.0, S_BELOW, 1.0]))]
    for attempt in range(4000):
        fid = fid0 + attempt
        d = _draws(fid, n, stream, call_no, offset, iters)
        hit = {x for ab in d for x in ab}
        free = [i for i in range(n) if i not in hit]
        if len(free) < k:
            continue
        rng = np.random.default_rng([fid, n, 6])
        T = _unit(np.array([rng.uniform(-0.5, 0.5), rng.uniform(-0.5, 0.5), 1.0]))
        ra, rb = np.empty((n, 3)), np.empty((n, 3))
        for i in range(n):
            ra[i], rb[i] = _scene_pair(rng, T, 3e-3, rng.uniform() < 0.2)
        special = [int(i) for i in rng.choice(free, k, replace=False)]
        for j, i in enumerate(special):
            ra[i], rb[i] = axes[j % 3]
        ts_a, ts_b = _timestamps(fid, n)
        f = Frame("e1", fid, ts_a, ts_b, ra, rb, stream, call_no, offset, iters, meta=dict(rows=special))
        v, q, best = f.trace(oracle_loader)
        P = oracle_problem(oracle_loader, [f]).problem_matrix(fid, 0.0, n)
        nP = P / np.linalg.norm(P, axis=1, keepdims=True)
        qn = np.partition((nP @ v.T) ** 2, n // 4, axis=0)[n // 4]
        alt = int(np.argmin(qn))
        if alt != best and sqrt_gap(qn, alt, best) > 4 * K_MARGIN:
            f.t1, f.t2 = best, alt
            return f
    raise AssertionError(f"no threshold-row frame for n={n}")
