"""An independent float64 restatement of the sparse pyramidal Lucas-Kanade tracker of
rssync_track_frames_device, written from the contract in include/rssync_b200.h (not from the kernels).

Differences from the engine are only those of the arithmetic: everything here is float64 and the window
sums are numpy sums, while the engine evaluates float32 in a stated order.  Each point also reports how
close it came to the two thresholds that decide its status (the eigenvalue test at every level, the image
border at the end), so a comparison can tell a real disagreement from one decided by rounding."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np


@dataclass
class Params:
    levels: int = 3
    window: int = 21
    max_iters: int = 30
    epsilon: float = 0.01
    min_eig: float = 1e-4


def pyr_down(img):
    """[1 4 6 4 1] / 16 blur with BORDER_REFLECT_101, every second row and column: size ((w + 1) // 2,
    (h + 1) // 2).  numpy's 'reflect' padding is BORDER_REFLECT_101 (the edge sample is not repeated)."""
    a = np.pad(np.asarray(img, dtype=np.float64), 2, mode="reflect")
    r = (a[:, :-4] + a[:, 4:]) + 4.0 * (a[:, 1:-3] + a[:, 3:-1]) + 6.0 * a[:, 2:-2]
    r = r[:, ::2]
    c = (r[:-4] + r[4:]) + 4.0 * (r[1:-3] + r[3:-1]) + 6.0 * r[2:-2]
    return c[::2] / 256.0


def pyramid(img, levels):
    out = [np.asarray(img, dtype=np.float64)]
    for _ in range(levels - 1):
        out.append(pyr_down(out[-1]))
    return out


def sample(level, x, y):
    """bilinear samples of `level` at float positions (arrays of one shape); integer reads are clamped to
    the level's edge"""
    h, w = level.shape
    x0, y0 = np.floor(x), np.floor(y)
    ax, ay = x - x0, y - y0
    xi, yi = x0.astype(np.int64), y0.astype(np.int64)

    def px(yy, xx):
        return level[np.clip(yy, 0, h - 1), np.clip(xx, 0, w - 1)]

    return ((1 - ay) * ((1 - ax) * px(yi, xi) + ax * px(yi, xi + 1)) +
            ay * ((1 - ax) * px(yi + 1, xi) + ax * px(yi + 1, xi + 1)))


def track(img_a, img_b, points, params=Params()):
    """Track points (n, 2) from img_a to img_b.  Returns a dict of arrays:
    tracked (n, 2; NaN where lost before the last level ended), status (bool), eig_margin (the smallest
    |min eigenvalue / min_eig - 1| over the levels evaluated), stop_margin (the smallest |delta^2 / epsilon^2
    - 1| over the iterations, 0 when a level used all max_iters: near 0, one more or one fewer iteration moves the result by up to ~epsilon)
    and border_margin (the tracked point's distance to the nearest border line of [0, w - 1] x [0, h - 1],
    signed: < 0 outside)."""
    p = params
    pts = np.asarray(points, dtype=np.float64).reshape(-1, 2)
    n = pts.shape[0]
    pa, pb = pyramid(img_a, p.levels), pyramid(img_b, p.levels)
    h0, w0 = pa[0].shape
    r, win = p.window // 2, p.window
    d = np.arange(-r - 1, r + 2, dtype=np.float64)
    DX, DY = np.meshgrid(d, d)  # (win + 2)^2 patch offsets, rows = dy
    fin = np.all(np.isfinite(pts), axis=1)
    ok = fin & (pts[:, 0] >= 0) & (pts[:, 0] <= w0 - 1) & (pts[:, 1] >= 0) & (pts[:, 1] <= h0 - 1)
    eig_margin = np.full(n, np.inf)
    stop_margin = np.full(n, np.inf)
    g = np.zeros((n, 2))
    v = np.zeros((n, 2))
    for lvl in range(p.levels - 1, -1, -1):
        idx = np.flatnonzero(ok)
        if idx.size == 0:
            break
        s = 2.0 ** -lvl
        q = pts[idx] * s
        A = sample(pa[lvl], q[:, 0, None, None] + DX, q[:, 1, None, None] + DY)  # (m, win + 2, win + 2)
        c = A[:, 1:-1, 1:-1]
        Ix = (3 * (A[:, :-2, 2:] - A[:, :-2, :-2]) + 10 * (A[:, 1:-1, 2:] - A[:, 1:-1, :-2]) +
              3 * (A[:, 2:, 2:] - A[:, 2:, :-2])) / 32.0
        Iy = (3 * (A[:, 2:, :-2] - A[:, :-2, :-2]) + 10 * (A[:, 2:, 1:-1] - A[:, :-2, 1:-1]) +
              3 * (A[:, 2:, 2:] - A[:, :-2, 2:])) / 32.0
        gxx, gxy, gyy = (Ix * Ix).sum((1, 2)), (Ix * Iy).sum((1, 2)), (Iy * Iy).sum((1, 2))
        min_eig = ((gxx + gyy) - np.sqrt((gxx - gyy) ** 2 + 4 * gxy ** 2)) / (2.0 * win * win)
        with np.errstate(divide="ignore", invalid="ignore"):
            eig_margin[idx] = np.minimum(eig_margin[idx], np.abs(min_eig / p.min_eig - 1.0))
        good = min_eig >= p.min_eig
        ok[idx[~good]] = False
        det = gxx * gyy - gxy * gxy
        vv = np.zeros((idx.size, 2))
        active = good.copy()
        inner = DX[1:-1, 1:-1], DY[1:-1, 1:-1]
        for _ in range(p.max_iters):
            ia = np.flatnonzero(active)
            if ia.size == 0:
                break
            bp = q[ia] + g[idx[ia]] + vv[ia]
            B = sample(pb[lvl], bp[:, 0, None, None] + inner[0], bp[:, 1, None, None] + inner[1])
            diff = c[ia] - B
            bx, by = (diff * Ix[ia]).sum((1, 2)), (diff * Iy[ia]).sum((1, 2))
            with np.errstate(divide="ignore", invalid="ignore"):
                ex = (gyy[ia] * bx - gxy[ia] * by) / det[ia]
                ey = (gxx[ia] * by - gxy[ia] * bx) / det[ia]
            bad = ~(np.isfinite(ex) & np.isfinite(ey))
            ok[idx[ia[bad]]] = False
            active[ia[bad]] = False
            upd = ~bad
            with np.errstate(invalid="ignore"):
                m = np.abs((ex * ex + ey * ey) / p.epsilon ** 2 - 1.0)
            stop_margin[idx[ia[upd]]] = np.minimum(stop_margin[idx[ia[upd]]], m[upd])
            vv[ia[upd], 0] += ex[upd]
            vv[ia[upd], 1] += ey[upd]
            done = upd & (ex * ex + ey * ey < p.epsilon ** 2)
            active[ia[done]] = False
        stop_margin[idx[active]] = 0.0  # max_iters reached: no stop decision to rely on
        keep = idx[ok[idx]]
        sel = ok[idx]
        if lvl > 0:
            g[keep] = 2.0 * (g[keep] + vv[sel])
        else:
            v[keep] = vv[sel]
    tracked = np.full((n, 2), np.nan)
    tracked[ok] = pts[ok] + g[ok] + v[ok]
    tx, ty = tracked[:, 0], tracked[:, 1]
    with np.errstate(invalid="ignore"):
        border = np.minimum(np.minimum(tx, w0 - 1 - tx), np.minimum(ty, h0 - 1 - ty))
        ok &= border >= 0
    return dict(tracked=tracked, status=ok, eig_margin=eig_margin, stop_margin=stop_margin, border_margin=border)
