"""An independent numpy restatement of the mask of rssync_track_frames_masked_device, written from the contract
in include/rssync_b200.h (not from the kernels): the eligibility of a pixel, the masked selection and the status
rule.  The scores, candidates and forward tracks come from the restatements in tests/select_reference.py and
tests/track_reference.py through their public functions."""
from __future__ import annotations

import numpy as np

import select_reference as sr
import track_reference as tr


def eligible(mask, margin):
    """(h, w) bool: pixel (x, y) is eligible iff every mask pixel within margin in x and in y that lies inside
    the image is nonzero (pixels outside count as usable).  Zeros counted in a (2 margin + 1) window along the
    rows, then along the columns, by prefix sums."""
    zero = np.asarray(mask) == 0
    margin = int(margin)

    def any_in_window(z, axis):
        z = np.moveaxis(z, axis, 0)
        c = np.concatenate([np.zeros((1,) + z.shape[1:], dtype=np.int64), np.cumsum(z, axis=0, dtype=np.int64)])
        n = z.shape[0]
        lo = np.clip(np.arange(n) - margin, 0, n)
        hi = np.clip(np.arange(n) + margin + 1, 0, n)
        return np.moveaxis((c[hi] - c[lo]) > 0, 0, axis)

    return ~any_in_window(any_in_window(zero, 1), 0)


def nearest(points):
    """the nearest pixel (floor(x + 0.5), floor(y + 0.5)) of (n, 2) double positions, as int64 (x, y)"""
    p = np.asarray(points, dtype=np.float64).reshape(-1, 2)
    return np.floor(p + 0.5).astype(np.int64)


def is_eligible(elig, points):
    """whether each position of (n, 2) points (inside the image) is eligible, at its nearest pixel"""
    q = nearest(points)
    return elig[q[:, 1], q[:, 0]]


def select(img, elig, opt=sr.Options(), score=None):
    """the masked selection of one image: select_reference's candidates that are also eligible, then the same
    cell picks, threshold (on the eligible picks' maximum) and max_points cut.  Returns (n, 2) float64 points in
    ascending cell order."""
    score = sr.scores(img, opt.block) if score is None else score
    h, w = score.shape
    cand = sr.candidates(score, opt.block) & np.asarray(elig, dtype=bool)
    ys, xs = np.nonzero(cand)
    sc = score[ys, xs]
    ncx = (w + opt.cell - 1) // opt.cell
    cell = (ys // opt.cell) * ncx + xs // opt.cell
    idx = ys.astype(np.int64) * w + xs
    order = np.lexsort((idx, -sc, cell))  # per cell: greatest score first, then the smallest index
    first = np.ones(order.size, dtype=bool)
    first[1:] = cell[order][1:] != cell[order][:-1]
    pick = order[first]
    pc, px, py, ps = cell[pick], xs[pick], ys[pick], sc[pick]
    kept = np.zeros(pick.size, dtype=bool)
    if pick.size:
        kept = ps >= np.float32(opt.quality) * ps.max()
        if kept.sum() > opt.max_points:
            k = np.flatnonzero(kept)
            best = k[np.lexsort((pc[k], -ps[k]))[:opt.max_points]]
            kept = np.zeros(pick.size, dtype=bool)
            kept[best] = True
    return np.stack([px[kept], py[kept]], axis=-1).astype(np.float64).reshape(-1, 2)


def masked_status(status, query, tracked, elig_a, elig_b):
    """the status rule: 3 where the unmasked forward status is 1 and the query point is not eligible on image i
    (elig_a) or the tracked position is not eligible on image i + 1 (elig_b); every other status unchanged"""
    st = np.asarray(status).astype(np.uint8).copy()
    one = np.flatnonzero(st == 1)
    if one.size:
        ok = is_eligible(elig_a, np.asarray(query)[one]) & is_eligible(elig_b, np.asarray(tracked)[one])
        st[one[~ok]] = 3
    return st


def track(img_a, img_b, query, elig_a, elig_b, params=tr.Params()):
    """the forward tracker restatement with the status rule applied: dict of track_reference.track plus
    masked (statuses 0, 1, 3)"""
    fwd = tr.track(img_a, img_b, query, params)
    fwd["masked"] = masked_status(fwd["status"], query, fwd["tracked"], elig_a, elig_b)
    return fwd
