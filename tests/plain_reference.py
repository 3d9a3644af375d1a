"""An independent restatement of rs-sync's loss chain in numpy ``longdouble``, for the tests.

The engine and the CPU oracle implement one arithmetic contract (DESIGN.md §3): FMA placement,
the ``log1p`` table, the folded quaternion normalisation, the RaySum order.  Comparing them with
each other cannot catch a formula that is wrong in the same way on both sides.  This module
restates the formulas from the reference (DESIGN.md §1 citations; the strict restatement in
``oracle/oracle_strict.hpp``; the simplified mode of ``include/rssync_b200.h``) without any of
those devices: plain numpy expressions, evaluated in ``np.longdouble`` (64-bit mantissa on x86),
rounded to float64 once at the end.  Inputs are float64.  Only two things are taken bit for bit
from the reference's own float64 arithmetic, because they are the reference's rounding and decide
*which* formula applies: the spline argument ``x = ((ts - q0) + delay) * sr`` and the pinned RNG.

Error bound
-----------
Every value is compared under a per-value first-order bound, not a flat tolerance.  With
``e = C * eps64`` (``C = 64``):

* a problem-matrix row is a cross product of two de-rotated unit rays: absolute error ``dP = e``
  per component (spline records, quaternion normalisation and the two rotations are each a few
  roundings of O(1) quantities);
* a hypothesis ``M`` is the normalised cross of two raw rows ``P_a x P_b``: its direction moves by
  ``dM = e * (1 + (|P_a| + |P_b|) / |P_a x P_b|)``, capped at 2 (two unit vectors are never
  further apart);
* ``P_i . M`` moves by ``d_i = dP + |P_i| dM``; ``|P M|`` by ``||d||_2 + depth * eps * |P M|``
  where ``depth = ceil(n / 32) + 5`` is the longest chain of additions of the 32-lane ray sum;
  ``k = clamp(1e2 / |P M|, 10, 1000)`` is monotone in ``|P M|``, so ``dk`` is its spread over
  ``|P M| +- d|P M|``;
* ``r_i = k (P_i . M) / |M|`` moves by ``dr_i = k d_i + |r_i| (dk / k + e)``;
* ``|d sqrt(log1p(r^2)) / dr| <= 1`` for every ``r`` (``log1p(r^2) >= r^2 / (1 + r^2)``), so a
  per-frame term moves by ``dr_i + e * term_i``; the sum ``S`` by the terms' bounds plus
  ``depth * eps * S``; and ``cost = sqrt(S)`` by ``dS / (sqrt(S) + sqrt(max(S - dS, 0)))``, which
  is exact for a square root and stays finite where ``S`` is rounding noise.

``Loss3`` (``|d log1p(r^2) / dr| <= 1``) and ``Loss5``'s gradient follow the same steps with ``m``
and ``k`` given.  A test asserts ``|engine - ref| <= bound`` and reports ``|engine - ref| / bound``.
Rounding differences give ratios far below 1; a wrong formula (a quartile rank, a constant, an
order) gives 10^6 or more.
"""
from __future__ import annotations

import numpy as np

LD = np.longdouble
EPS = float(np.finfo(np.float64).eps)
C_BOUND = 64
E = C_BOUND * EPS
MASK = (1 << 64) - 1

# ------------------------------------------------------------------------------------------------
# pinned RNG (DESIGN.md §3.6), in Python integers


def mix64(z):
    z &= MASK
    z ^= z >> 30
    z = (z * 0xBF58476D1CE4E5B9) & MASK
    z ^= z >> 27
    z = (z * 0x94D049BB133111EB) & MASK
    z ^= z >> 31
    return z


def rng_prefix(seed, stream, call_no, offset_idx):
    h = mix64(seed + 0x9E3779B97F4A7C15)
    h = mix64(h ^ ((stream + (call_no << 8)) & MASK))
    return mix64(h ^ (offset_idx & MASK))


def rng_task_key(seed, stream, call_no, offset_idx, frame_id):
    return mix64(rng_prefix(seed, stream, call_no, offset_idx) ^ (int(frame_id) & MASK))


def rng_index(key, it, k, n):
    """mulhi64(mix64(key ^ (iter << 32 | k)), n)"""
    return (mix64(key ^ ((it << 32) | k)) * n) >> 64


def draws(key, iters, n):
    """the estimator's row pairs: a, then b != a (core_private.cpp:42-43)"""
    out = []
    for it in range(iters):
        a = rng_index(key, it, 0, n)
        k = 1
        while True:
            b = rng_index(key, it, k, n)
            k += 1
            if b != a:
                break
        out.append((a, b))
    return out


# ------------------------------------------------------------------------------------------------
# spline and rows


def spline_x(ts, q0, sr, delay):
    """the spline argument in the reference's own float64 rounding (core_private.cpp:19-20)"""
    ts = np.asarray(ts, dtype=np.float64)
    return ((ts - np.float64(q0)) + np.float64(delay)) * np.float64(sr)


def spline_eval(rec, x):
    """spline::operator() (minispline.cpp:48-55) from {y, b, c, d} records, all four components:
    linear on the left (c[0] = 0), the last record's quadratic on the right with
    h = x - min(floor(x), n) (a sawtooth at x >= n), Horner inside.  -> (len(x), 4) longdouble"""
    rec = np.asarray(rec, dtype=np.float64)
    n = rec.shape[0]
    x = np.asarray(x, dtype=np.float64)
    fl = np.floor(x)
    idx = np.clip(fl, 0.0, float(n))
    h = (x.astype(LD) - idx.astype(LD))[:, None]
    R = rec.astype(LD)
    y, b, c, d = R[:, 0:4], R[:, 4:8], R[:, 8:12], R[:, 12:16]
    left = x < idx
    right = x > n - 1
    i = np.minimum(idx.astype(np.int64), n - 1)
    inner = ((d[i] * h + c[i]) * h + b[i]) * h + y[i]
    out = inner
    out = np.where(right[:, None], (c[n - 1] * h + b[n - 1]) * h + y[n - 1], out)
    out = np.where(left[:, None], (c[0] * h + b[0]) * h + y[0], out)
    return out


def qprod(p, q):
    """Hamilton product of (..., 4) arrays (quat.cpp:33-38)"""
    p0, p1, p2, p3 = p[..., 0], p[..., 1], p[..., 2], p[..., 3]
    q0, q1, q2, q3 = q[..., 0], q[..., 1], q[..., 2], q[..., 3]
    return np.stack([p0 * q0 - p1 * q1 - p2 * q2 - p3 * q3,
                     p0 * q1 + p1 * q0 + p2 * q3 - p3 * q2,
                     p0 * q2 - p1 * q3 + p2 * q0 + p3 * q1,
                     p0 * q3 + p1 * q2 - p2 * q1 + p3 * q0], axis=-1)


def derotate(q, p):
    """quat_rotate_point(conj(q / |q|), p) = conj(q) (x) (0, p) (x) q with q normalised"""
    q = q / np.sqrt(np.sum(q * q, axis=-1, keepdims=True))
    pq = np.concatenate([np.zeros(p.shape[:-1] + (1,), dtype=LD), p], axis=-1)
    conj = q * np.array([1, -1, -1, -1], dtype=LD)
    return qprod(conj, qprod(pq, q))[..., 1:]


def rows(rec, q0, sr, delay, ts_a, ts_b, rays_a, rays_b):
    """opt_compute_problem (core_private.cpp:15-32): one row per ray pair, caller order, longdouble"""
    qa = spline_eval(rec, spline_x(ts_a, q0, sr, delay))
    qb = spline_eval(rec, spline_x(ts_b, q0, sr, delay))
    ar = derotate(qa, np.asarray(rays_a, dtype=np.float64).astype(LD))
    br = derotate(qb, np.asarray(rays_b, dtype=np.float64).astype(LD))
    return np.cross(ar, br)


def frame_rows(rec, q0, sr, delay, w, i, n=None):
    """rows of frame index i of a synth.Workload (first n rays)"""
    n = w.ts_a.shape[1] if n is None else n
    return rows(rec, q0, sr, delay, w.ts_a[i, :n], w.ts_b[i, :n], w.rays_a[i, :n], w.rays_b[i, :n])


def span_edge_delays(w, i, nq):
    """delays that put frame i's rays across the first knot, across the last knot, on an exact
    integer x, inside [nq - 1, nq) and at x >= nq"""
    lo, hi = float(np.min(w.ts_a[i])), float(np.max(w.ts_a[i]))
    mid = float(np.median(w.ts_a[i]))
    t_last = w.gyro_t0 + (nq - 1) / w.gyro_rate
    d_int = spline_x([mid], w.gyro_t0, w.gyro_rate, 0.0)[0]
    return np.array([
        w.gyro_t0 - mid,                     # first knot inside the frame's readout
        w.gyro_t0 - hi - 0.002,              # every ray left of the first knot
        t_last - mid,                        # last knot inside the readout
        t_last - lo + 0.0005,                # every ray in [nq - 1, nq) or beyond
        t_last - lo + 1.5 / w.gyro_rate,     # x >= nq: the sawtooth
        (np.ceil(d_int) - d_int) / w.gyro_rate,  # the median ray near an integer x
    ])


# ------------------------------------------------------------------------------------------------
# estimator, k, losses

TIE_REL = 1e-9
TIE_FLOOR = (64 * EPS) ** 2


def safe_normalize(v):
    """inline_utils.hpp:5-11: vectors of norm < 1e-12 are left as they are"""
    nrm = np.sqrt(np.sum(v * v, axis=-1, keepdims=True))
    return np.where(nrm < 1e-12, v, v / np.where(nrm < 1e-12, 1, nrm))


class Estimate:
    """opt_guess_translational_motion (core_private.cpp:34-59) with every hypothesis kept"""

    def __init__(self, P, key, iters, row_err=0.0):
        n = P.shape[0]
        self.pairs = draws(key, iters, n)
        a = np.array([p[0] for p in self.pairs])
        b = np.array([p[1] for p in self.pairs])
        raw = np.cross(P[a], P[b])
        self.raw_norm = np.sqrt(np.sum(raw * raw, axis=1))
        self.hyp = safe_normalize(raw)                           # :45-46
        nP = safe_normalize(P)                                   # :35-36
        r2 = (nP @ self.hyp.T) ** 2                              # :48-49, (n, iters)
        self.quartile = np.partition(r2, n // 4, axis=0)[n // 4]  # :51-52
        best = 0
        for t in range(1, iters):                                # :53-56, strict <
            if self.quartile[t] < self.quartile[best]:
                best = t
        self.best = best
        qb = self.quartile[best]
        self.near = [t for t in range(iters)
                     if self.quartile[t] - qb <= TIE_REL * qb or self.quartile[t] <= TIE_FLOOR]
        row_norm = np.sqrt(np.sum(P * P, axis=1))
        row_err = np.broadcast_to(np.asarray(row_err, dtype=np.float64), (n,))
        raw = np.maximum(self.raw_norm.astype(np.float64), 1e-300)
        self.dM = np.minimum(2.0, E * (1.0 + (row_norm[a] + row_norm[b]).astype(np.float64) / raw)
                             + (row_err[a] + row_err[b]) / raw)

    def distinct_near(self):
        """near-tie members with distinct hypotheses (index of the first of each)"""
        out, seen = [], []
        for t in self.near:
            h = tuple(float(x) for x in self.hyp[t])
            if h not in seen:
                seen.append(h)
                out.append(t)
        return out


def clamp_k(k):
    """std::clamp(k, 1e1, 1e3) (inline_utils.hpp:50)"""
    return np.minimum(np.maximum(k, LD(10)), LD(1000))


def depth(n):
    return (n + 31) // 32 + 5


def k_of(P, M):
    """GuessK: clamp(1e2 / ||P M||)  (core_private.cpp:79, :132)"""
    return clamp_k(LD(100) / np.sqrt(np.sum((P @ M) ** 2)))


def _k_spread(N, dN):
    lo = clamp_k(LD(100) / max(N - dN, LD(0))) if N - dN > 0 else LD(1000)
    return float(lo - clamp_k(LD(100) / (N + dN)))


def _sqrt_bound(S, dS):
    den = np.sqrt(S) + np.sqrt(max(S - dS, 0.0))
    return dS / den if den > 0 else np.sqrt(dS)


def presync_cost(P, M=None, dM=0.0, simplified=False, row_err=0.0):
    """per-frame body of pre_sync (core_private.cpp:75-85): k = clamp(1e2 / ||P M||),
    r = P M k / |M|, cost = sqrt(sum sqrt(log1p(r^2))).  Simplified mode (include/rssync_b200.h):
    the residual of a ray is its row's norm.  row_err: an absolute error of each row (per row or one
    for all) on top of the rows' own rounding, e.g. from rays that are themselves approximations.
    -> (cost, bound, k, bound of k)"""
    n = P.shape[0]
    rn = np.sqrt(np.sum(P * P, axis=1))
    row_err = np.broadcast_to(np.asarray(row_err, dtype=np.float64), (n,))
    if simplified:
        v = rn
        d = E + row_err
        scale_div = LD(1)
    else:
        v = P @ M
        d = E + row_err + rn.astype(np.float64) * dM
        scale_div = np.sqrt(np.sum(M * M))
    N = np.sqrt(np.sum(v * v))
    with np.errstate(divide="ignore"):
        k = clamp_k(LD(100) / N)  # 1e2 / 0 = inf -> 1000, as in the reference
    dN = float(np.sqrt(np.sum(d * d))) + depth(n) * EPS * float(N)
    dk = _k_spread(N, LD(dN))
    with np.errstate(invalid="ignore", divide="ignore"):
        r = v * (k / scale_div)
        term = np.sqrt(np.log1p(r * r))
    S = np.sum(term)
    cost = np.sqrt(S)
    kf = float(k)
    dr = kf * d + np.abs(r.astype(np.float64)) * (dk / kf + E)
    dS = float(np.sum(dr + E * term.astype(np.float64))) + depth(n) * EPS * float(S)
    return float(cost), _sqrt_bound(float(S), dS) + EPS * float(cost), kf, dk + E * kf


def presync_cell(P, key=None, simplified=False, iters=20, row_err=0.0):
    """one (delay, frame) cell of the PreSync grid: the frame's cost for every near-tie hypothesis
    of the estimator -> list of (cost, bound).  row_err: as in presync_cost"""
    if simplified:
        c, b, _, _ = presync_cost(P, simplified=True, row_err=row_err)
        return [(c, b)]
    est = Estimate(P, key, iters, row_err)
    return [presync_cost(P, est.hyp[t], float(est.dM[t]), row_err=row_err)[:2] for t in est.distinct_near()]


def cell_ratio(got, cands):
    """|got - ref| / bound against the closest candidate"""
    return min(ratio(got, c, b) for c, b in cands)


def loss3(P, m, k):
    """FrameState::Loss, 3 arguments (core_private.cpp:117-123) -> (value, bound)"""
    m = np.asarray(m, dtype=np.float64).astype(LD)
    kk = LD(float(k))
    r = (P @ m) * (kk / np.sqrt(np.sum(m * m)))
    t = np.log1p(r * r)
    dr = float(kk) * E + np.abs(r.astype(np.float64)) * E
    L = np.sum(t)
    return float(L), float(np.sum(dr + E * t.astype(np.float64))) + depth(P.shape[0]) * EPS * float(L)


def loss5(P, m, k):
    """FrameState::Loss, 5 arguments (core_private.cpp:92-115): the value and the closed-form
    gradient d/dm of sum log1p(u_i), u_i = (P_i.m)^2 k^2 / |m|^2 -> (value, grad, value bound,
    gradient bound per component)"""
    n = P.shape[0]
    m = np.asarray(m, dtype=np.float64).astype(LD)
    kk = LD(float(k))
    mn2 = np.sum(m * m)
    den = mn2 / (kk * kk)
    v1 = P @ m
    u = v1 * v1 / den
    L = np.sum(np.log1p(u))
    w = 1 / (1 + u)
    terms = w[:, None] * ((2 * v1 / den)[:, None] * P - ((v1 * v1) / (den * den) / (kk * kk))[:, None] * (2 * m))
    g = np.sum(terms, axis=0)
    _, dL = loss3(P, m, k)
    # each term is (2 / (|m| (1 + r^2))) (k r P_i - r^2 m/|m|) with r = k P_i.m / |m|
    mn = float(np.sqrt(mn2))
    r = np.abs((v1 * kk / np.sqrt(mn2)).astype(np.float64))
    rn = np.sqrt(np.sum(P * P, axis=1)).astype(np.float64)
    kf = float(kk)
    dr = kf * E + r * E
    dt = ((2.0 / mn) * ((kf * rn + 1.0) * dr + kf * E))[:, None] + E * np.abs(terms.astype(np.float64))
    dg = np.sum(dt, axis=0) + depth(n) * EPS * np.sum(np.abs(terms.astype(np.float64)), axis=0)
    return float(L), g.astype(np.float64), dL, dg


def rows_bound(P):
    """absolute bound per row component"""
    return np.full(P.shape, E)


def ratio(got, want, bound):
    """largest |got - want| / bound (0 where both are equal)"""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    bound = np.broadcast_to(np.asarray(bound, dtype=np.float64), want.shape)
    diff = np.abs(got - want)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(diff == 0, 0.0, diff / bound)
    return float(np.max(r)) if r.size else 0.0


class RatioLog:
    """largest bound ratio seen per stage (printed by the tests, -s)"""

    def __init__(self):
        self.worst = {}

    def add(self, stage, r):
        self.worst[stage] = max(self.worst.get(stage, 0.0), float(r))
        return r

    def report(self):
        return ", ".join(f"{k} {v:.3g}" for k, v in sorted(self.worst.items()))
