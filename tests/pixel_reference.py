"""An independent restatement of the pixel -> ray front end (rssync_set_track_pixels: lens_undistort_point,
core_testcode.cpp:63-95, the rolling-shutter timestamps :144-145 and the unit rays :147-154) and of the way
the engine stores a frame (ingest_sort_and_store, engine.cu), for the tests.

It follows the rules of ``plain_reference``: plain numpy, no engine code.  Only the values of the
reference's own float64 arithmetic that decide *which* formula applies are taken bit for bit from
float64:

* the Newton iteration for theta.  It uses +, -, *, / and comparisons only, here in the kernel's order;
  the library is built with ``-fmad=false``, so this replay gives the engine's exact theta, the halvings
  that keep it inside (0, pi/2) and the 2048-round guard included;
* the branch decisions ``|p| < 1e-8`` (raw pixel: the optical axis) and ``theta_ < 1e-9`` (``1 / cos``
  instead of ``tan / theta_``);
* the timestamps ``frame_ts + readout * (y / rows)``, which are stored and sorted on.

Everything after theta -- ``tan``, ``1 / cos``, the scale ``s``, the normalisation of (x', y', 1) -- is
evaluated in ``np.longdouble`` and rounded once.  Where the float64 iteration converged, theta is also
solved independently: the root of theta (1 + k1 theta^2 + k2 theta^4 + k3 theta^6 + k4 theta^8) = theta_d,
bisected in long double on (0, pi/2); the reference ray uses that root, which checks that the iteration
lands on the model's root (a swapped or misplaced coefficient does not).  Where it did not converge (far
outside the image circle, strong lenses) the replayed theta *is* the reference's answer, and that is the
only place where its derivative coefficient ``8 k4`` (the exact one is ``9 k4``) shows.

Error bound
-----------
A ray's angle from the optical axis is theta, so rays are compared by the angle between engine and
reference ray, not by components (near pi/2 tan is huge, the angle is not).  With ``e = C * eps64``
(``C = 64``, as in ``plain_reference``): on converged points ``e * (1 + theta_d / f'(theta))`` with the
long-double root and the true derivative f' (a relative rounding of theta_d moves the root by
``theta_d eps / f'``); on replayed points ``e``, which also covers CUDA's tan / cos (<= 2 ulp).

Deliberate deviation from ``synth.undistort``: that restatement has no raw-pixel check (core_testcode.cpp
:64), so (0, 0) and points within 1e-8 of it get an ordinary ray there and the optical axis here.  The
synthetic workloads never come near it, and ``synth`` generates them, so it stays as it is.
"""
from __future__ import annotations

import numpy as np

from plain_reference import E, EPS, LD

K_PI = 3.14159265358979323846  # the kernel's kPi, a float64
GUARD = 2048
CONVERGED_STEP = 16 * EPS  # a last Newton step below this (relative to theta): converged


class Lens:
    """rssync_lens field order: readout, fx, fy, cx, cy, k1, k2, k3, k4"""

    def __init__(self, readout, fx, fy, cx, cy, k1, k2, k3, k4):
        self.readout, self.fx, self.fy, self.cx, self.cy = (float(v) for v in (readout, fx, fy, cx, cy))
        self.k = tuple(float(v) for v in (k1, k2, k3, k4))

    def tuple(self, readout=None):
        return (self.readout if readout is None else float(readout), self.fx, self.fy, self.cx, self.cy) + self.k


def newton(theta_d, k, k4_coef=8.0, steps=9):
    """the kernel's float64 iteration from pi/4, vectorised -> (theta, last step, halvings)"""
    k1, k2, k3, k4 = k
    theta_d = np.asarray(theta_d, dtype=np.float64)
    th = np.full(theta_d.shape, K_PI / 4.0)
    halv = np.zeros(theta_d.shape, dtype=np.int64)
    last = np.zeros(theta_d.shape)
    with np.errstate(all="ignore"):
        for _ in range(steps):
            t2 = th * th
            t3 = t2 * th
            t4 = t2 * t2
            t5 = t2 * t3
            t6 = t3 * t3
            t7 = t3 * t4
            t8 = t4 * t4
            t9 = t4 * t5
            cur = th + k1 * t3 + k2 * t5 + k3 * t7 + k4 * t9
            dcur = 1 + 3 * k1 * t2 + 5 * k2 * t4 + 7 * k3 * t6 + k4_coef * k4 * t8
            err = cur - theta_d
            nt = th - err * (1.0 / dcur)
            for _g in range(GUARD):
                out = (nt >= K_PI / 2.0) | (nt <= 0.0)
                if not out.any():
                    break
                nt = np.where(out, (nt + th) / 2.0, nt)
                halv += out
            last = nt - th
            th = nt
    return th, last, halv


def poly(theta, k):
    k1, k2, k3, k4 = (LD(v) for v in k)
    t2 = theta * theta
    return theta * (1 + t2 * (k1 + t2 * (k2 + t2 * (k3 + t2 * k4))))


def dpoly(theta, k):
    """the true derivative (coefficient 9 k4)"""
    k1, k2, k3, k4 = (LD(v) for v in k)
    t2 = theta * theta
    return 1 + t2 * (3 * k1 + t2 * (5 * k2 + t2 * (7 * k3 + t2 * 9 * k4)))


def root(theta_d, k):
    """theta in (0, pi/2) with poly(theta) = theta_d, bisected in long double; NaN without a sign change"""
    td = np.asarray(theta_d, dtype=np.float64).astype(LD)
    lo = np.zeros(td.shape, dtype=LD)
    hi = np.full(td.shape, LD(np.pi) / 2)
    ok = (poly(hi, k) - td > 0) & (td > 0)
    for _ in range(80):
        mid = (lo + hi) / 2
        below = poly(mid, k) - td < 0
        lo = np.where(below, mid, lo)
        hi = np.where(below, hi, mid)
    return np.where(ok, (lo + hi) / 2, LD(np.nan))


class Undistorted:
    """the reference's rays of points (n, 2) through `lens`.  Fields (per point): ray (n, 3) long double,
    bound (angle, radians), axis (the raw-pixel check fired), theta_d, theta (float64 replay), halvings,
    converged, small (the 1 / cos branch)"""

    def __init__(self, pts, lens, k4_coef=8.0):
        pts = np.asarray(pts, dtype=np.float64).reshape(-1, 2)
        px, py = pts[:, 0], pts[:, 1]
        with np.errstate(all="ignore"):
            self.axis = np.sqrt(px * px + py * py) < 1e-8
            x_ = (px - lens.cx) / lens.fx
            y_ = (py - lens.cy) / lens.fy
            self.theta_d = np.sqrt(x_ * x_ + y_ * y_)
        self.theta, last, self.halvings = newton(self.theta_d, lens.k, k4_coef)
        self.small = self.theta_d < 1e-9
        self.converged = (np.abs(last) <= CONVERGED_STEP * self.theta) & (self.theta_d > 0) & ~self.axis
        th = self.theta.astype(LD)
        rt = root(np.where(self.converged, self.theta_d, 1.0), lens.k)
        self.root_missing = self.converged & np.isnan(rt)
        th = np.where(self.converged & ~self.root_missing, rt, th)
        self.theta_ref = th
        with np.errstate(all="ignore"):
            s = np.where(self.small, 1 / np.cos(th), np.tan(th) / np.where(self.small, 1.0, self.theta_d).astype(LD))
            ux = x_.astype(LD) * s
            uy = y_.astype(LD) * s
            ux = np.where(self.axis, LD(0), ux)
            uy = np.where(self.axis, LD(0), uy)
            nrm = np.sqrt(ux * ux + uy * uy + 1)
        self.ray = np.stack([ux / nrm, uy / nrm, 1 / nrm], axis=-1)
        fp = dpoly(th, lens.k).astype(np.float64)
        with np.errstate(all="ignore"):
            conv_bound = E * (1.0 + self.theta_d / fp)
        self.bound = np.where(self.converged, conv_bound, E)


def angle(a, b):
    """angle (radians, float64) between rays a and b (n, 3), evaluated in long double"""
    a = np.asarray(a).astype(LD)
    b = np.asarray(b).astype(LD)
    c = np.cross(a, b)
    return np.arctan2(np.sqrt(np.sum(c * c, axis=-1)), np.sum(a * b, axis=-1)).astype(np.float64)


def angle_ratio(got, und):
    """largest angle(got, reference) / bound over the points"""
    ang = angle(got, und.ray)
    return float(np.max(np.where(ang == 0, 0.0, ang / und.bound))) if ang.size else 0.0


def _tiles(flat):
    """(8, padded) field x slot -> the arena's tiles (padded / 32, 8, 32)"""
    return np.ascontiguousarray(flat.reshape(8, -1, 32).transpose(1, 0, 2))


def timestamps(frame_ts, y, readout, rows):
    """frame_ts + readout * (y / rows), the reference's float64 rounding (core_testcode.cpp:144-145)"""
    return np.float64(frame_ts) + np.float64(readout) * (np.asarray(y, dtype=np.float64) / np.float64(rows))


class Frame:
    """what the engine stores for one frame of pixel pairs: ts_a, ts_b (caller order), the rays of both
    sides (Undistorted), the storage order (sorted by (ts_a, caller index)), the tiles
    [ceil(n / 32)][8 fields][32 lanes] (ts_a, ts_b, ray a xyz, ray b xyz), the orig / pos planes and
    the frame table's ts_lo / ts_hi"""

    def __init__(self, pa, pb, frame_ts_a, frame_ts_b, lens, rows, readout=None, und=None):
        pa = np.asarray(pa, dtype=np.float64).reshape(-1, 2)
        pb = np.asarray(pb, dtype=np.float64).reshape(-1, 2)
        self.n = n = pa.shape[0]
        ro = lens.readout if readout is None else float(readout)
        self.ts_a = timestamps(frame_ts_a, pa[:, 1], ro, rows)
        self.ts_b = timestamps(frame_ts_b, pb[:, 1], ro, rows)
        self.und_a, self.und_b = und if und is not None else (Undistorted(pa, lens), Undistorted(pb, lens))
        self.order = np.lexsort((np.arange(n), self.ts_a))  # ts_a, ties by caller index
        padded = (n + 31) // 32 * 32
        self.orig = np.arange(padded, dtype=np.int32)
        self.orig[:n] = self.order
        self.pos = np.arange(padded, dtype=np.int32)
        self.pos[self.order] = np.arange(n, dtype=np.int32)
        flat = np.zeros((8, padded))  # field, slot
        ra = self.und_a.ray.astype(np.float64)
        rb = self.und_b.ray.astype(np.float64)
        fields = [self.ts_a, self.ts_b, ra[:, 0], ra[:, 1], ra[:, 2], rb[:, 0], rb[:, 1], rb[:, 2]]
        for c, v in enumerate(fields):
            flat[c, :n] = v[self.order]
        if n:
            flat[0, n:] = self.ts_a[self.order[-1]]  # padding: the last ray's timestamps, zeros elsewhere
            flat[1, n:] = self.ts_b[self.order[-1]]
        self.tiles = _tiles(flat)
        both = np.concatenate([self.ts_a, self.ts_b])
        self.ts_lo = float(both.min()) if n else 0.0
        self.ts_hi = float(both.max()) if n else 0.0

    def retimed(self, pa, pb, frame_ts_a, frame_ts_b, lens, rows, readout):
        """the same frame at another readout (its rays are not recomputed)"""
        return Frame(pa, pb, frame_ts_a, frame_ts_b, lens, rows, readout, (self.und_a, self.und_b))

    def ray_mask(self):
        """tile positions that hold ray components of real rays (fields 2..7, slots < n)"""
        flat = np.zeros((8, self.tiles.shape[0] * 32), dtype=bool)
        flat[2:, :self.n] = True
        return _tiles(flat)

    def ray_bounds(self):
        """per caller ray: the angle bounds of side a and side b"""
        return self.und_a.bound, self.und_b.bound
