"""An independent float32 restatement of the point selection of rssync_track_frames_ex_device, written from the
contract in include/rssync_b200.h (not from the kernels), and the forward-backward check composed from the
tracker restatement (tests/track_reference.py).

The selection has no float64 step and no reduction of variable order, and numpy neither contracts into FMA nor
rounds np.sqrt differently from a correctly rounded sqrtf, so the scores, picks and points here equal the
engine's bit for bit.  Every sum is written out term by term, in the contract's order."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

import track_reference as tr


@dataclass
class Options:
    cell: int = 128
    block: int = 5
    quality: float = 0.01
    max_points: int = 512
    fb_max: float = 1.0


def scores(img, block):
    """the minimum eigenvalue of the structure tensor of every pixel, float32 (cv2.cornerMinEigenVal(img, block, 3));
    numpy's 'reflect' padding is BORDER_REFLECT_101"""
    f = np.asarray(img).astype(np.float32)
    p = np.pad(f, 1, mode="reflect")
    s = np.float32(1.0 / (4 * block * 255))
    two = np.float32(2.0)
    dx = (((p[:-2, 2:] - p[:-2, :-2]) + two * (p[1:-1, 2:] - p[1:-1, :-2])) + (p[2:, 2:] - p[2:, :-2])) * s
    dy = (((p[2:, :-2] - p[:-2, :-2]) + two * (p[2:, 1:-1] - p[:-2, 1:-1])) + (p[2:, 2:] - p[:-2, 2:])) * s
    r = block // 2
    H, W = f.shape

    def box(a):
        q = np.pad(a, r, mode="reflect")
        rows = q[:, 0:W]
        for i in range(1, block):  # each row left to right
            rows = rows + q[:, i:i + W]
        out = rows[0:H]
        for i in range(1, block):  # then the row sums top to bottom
            out = out + rows[i:i + H]
        return out

    xx, xy, yy = box(dx * dx), box(dx * dy), box(dy * dy)
    a, c = np.float32(0.5) * xx, np.float32(0.5) * yy
    d = a - c
    return (a + c) - np.sqrt(d * d + xy * xy)


def candidates(score, block):
    """boolean map of the candidates: inside the margin block / 2 + 2, score > 0, >= its 8 neighbours"""
    h, w = score.shape
    m = block // 2 + 2
    out = np.zeros((h, w), dtype=bool)
    if h - 2 * m <= 0 or w - 2 * m <= 0:
        return out
    c = score[m:h - m, m:w - m]
    ok = c > 0
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            if dy or dx:
                ok &= c >= score[m + dy:h - m + dy, m + dx:w - m + dx]
    out[m:h - m, m:w - m] = ok
    return out


def select(img, opt=Options(), score=None):
    """the selected points of one image: dict with points ((n, 2) float64, ascending cell order), and for
    inspection score (the score map), picks (every cell's pick: cell, x, y, score) and kept (bool per pick).
    score: scores(img, opt.block) when already computed"""
    score = scores(img, opt.block) if score is None else score
    h, w = score.shape
    cand = candidates(score, opt.block)
    ys, xs = np.nonzero(cand)
    sc = score[ys, xs]
    ncx = (w + opt.cell - 1) // opt.cell
    cell = (ys // opt.cell) * ncx + xs // opt.cell
    idx = ys.astype(np.int64) * w + xs
    order = np.lexsort((idx, -sc, cell))  # per cell: greatest score first, then the smallest index
    first = np.ones(order.size, dtype=bool)
    first[1:] = cell[order][1:] != cell[order][:-1]
    pick = order[first]  # ascending cell order
    pc, px, py, ps = cell[pick], xs[pick], ys[pick], sc[pick]
    kept = np.zeros(pick.size, dtype=bool)
    if pick.size:
        thr = np.float32(opt.quality) * ps.max()
        kept = ps >= thr
        if kept.sum() > opt.max_points:
            k = np.flatnonzero(kept)
            best = k[np.lexsort((pc[k], -ps[k]))[:opt.max_points]]  # greatest score, then the smaller cell
            kept = np.zeros(pick.size, dtype=bool)
            kept[best] = True
    points = np.stack([px[kept], py[kept]], axis=-1).astype(np.float64).reshape(-1, 2)
    return dict(points=points, score=score, kept=kept,
                picks=dict(cell=pc, x=px, y=py, score=ps))


def forward_backward(img_a, img_b, points, params=tr.Params(), fb_max=1.0):
    """the forward pass, then (fb_max > 0) the backward pass of the points it kept: dict with forward (the
    forward track_reference result), u (the backward result, NaN where not run or lost), fb (NaN where the
    backward pass did not keep the point) and status (0 lost, 1 kept, 2 rejected by the backward check)"""
    q = np.asarray(points, dtype=np.float64).reshape(-1, 2)
    fwd = tr.track(img_a, img_b, q, params)
    st = fwd["status"]
    n = q.shape[0]
    u = np.full((n, 2), np.nan)
    fb = np.full(n, np.nan)
    status = st.astype(np.uint8)
    bwd = None
    if fb_max > 0 and st.any():
        bwd = tr.track(img_b, img_a, fwd["tracked"][st], params)
        k = np.flatnonzero(st)
        u[k] = bwd["tracked"]
        back = bwd["status"]
        d = u[k] - q[k]
        f = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1])
        fb[k[back]] = f[back]
        with np.errstate(invalid="ignore"):
            status[k] = np.where(back & (fb[k] <= fb_max), 1, 2)
    return dict(forward=fwd, backward=bwd, u=u, fb=fb, status=status)
