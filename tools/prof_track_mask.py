"""Measure the cost of a caller's mask in device tracking (rssync_track_frames_masked_device), on 64 frames of
rendered luma planes (tests/render_reference.py) at 2704 x 2028 and 3840 x 2160, with selection and the backward
check on (TrackOptions defaults: 128-px cells, block 5, 512 points, fb_max 1 px) and the default margin (11 px).

  (a) per call of 64 frames, median and p10-p90 of a host clock around the call ending in a synchronise, the
      three cases alternating: no mask (rssync_track_frames_ex_device), a shared mask (96-px bands at the top
      and bottom, an OSD), and per-image masks (the bands plus a 300-px square moving 16 px per image);
  (b) per-kernel times of each case from torch.profiler, in a separate pass;
  (c) with --base-lib (a build of the parent commit): the unmasked path at 2704 x 2028 through this build and
      through the base build, alternating in subprocesses over plain ctypes; the outputs and frame tables must
      be bit-identical.

The card's name, power limit and max SM clock are read in the same run.  Writes prof_track_mask.json to --out."""
from __future__ import annotations

import argparse
import importlib
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import prof_track16 as pt  # noqa: E402  (the clip, the statistics, the GPU identification, the base-build child)

KERNELS = ("track_erode_kernel",) + pt.KERNELS
SIZES = ((2704, 2028), (3840, 2160))


def _masks(w, h, n, device):
    import torch
    shared = torch.ones((h, w), dtype=torch.uint8, device=device)
    shared[:96] = 0
    shared[-96:] = 0
    per = shared.repeat(n, 1, 1)
    for j in range(n):
        x0, y0 = 200 + 16 * j, h // 3
        per[j, y0:y0 + 300, x0:x0 + 300] = 0
    return shared, per


def timing(w, h, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    rsb = importlib.import_module("rs-sync_b200")
    clip, imgs = pt._clip(w, h)
    shared, per = _masks(w, h, clip.n_images, "cuda:0")
    ids, ts, lens = clip.frame_ids(), clip.image_ts(), clip.lens()
    opt = rsb.TrackOptions()

    def problem():
        p = rsb.SyncProblem(seed=100)
        p.SetGyroQuaternions(clip.quats, clip.quats.shape[0], clip.gyro_rate, clip.gyro_t0)
        return p

    cases = {
        "no_mask": lambda p: p.track_frames_ex(ids, ts, imgs, lens, options=opt),
        "shared_mask": lambda p: p.track_frames_ex(ids, ts, imgs, lens, options=opt, mask=shared),
        "per_image_masks": lambda p: p.track_frames_ex(ids, ts, imgs, lens, options=opt, mask=per),
    }
    ms = {k: [] for k in cases}
    res = {}
    for i in range(reps + 1):
        for name, call in cases.items():
            p = problem()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = call(p)
            torch.cuda.synchronize()
            if i:
                ms[name].append((time.perf_counter() - t0) * 1e3)
            res[name] = r
    out = {}
    for name, call in cases.items():
        call(problem())
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                call(problem())
            torch.cuda.synchronize()
        kt = {}
        for e in prof.key_averages():
            m = re.search(r"(%s)(<[^>]*>)?" % "|".join(KERNELS), e.key)
            if m:  # keyed by the name with its template arguments
                key = m.group(0)
                kt[key] = kt.get(key, 0.0) + e.device_time_total / 1e3 / reps  # ms per call
        st = res[name].status
        out[name] = {"frames_per_call": 64, "points": int(st.numel()),
                     "status_counts": {str(v): int((st == v).sum()) for v in (0, 1, 2, 3)},
                     "call_ms": pt._stats(ms[name]), "kernel_ms_per_call": kt,
                     "kernel_ms_sum": float(sum(kt.values()))}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--base-lib", default=None)
    a = ap.parse_args()
    res = {"gpu": pt.gpu_info()}
    for w, h in SIZES:
        res[f"frames_{w}x{h}"] = timing(w, h, a.reps)
    res["no_mask_vs_base"] = "not measured (no --base-lib)"
    if a.base_lib:
        libs = {"this": os.path.join(ROOT, "rs-sync_b200", "lib", "librssync_b200.so"), "base": a.base_lib}
        runs = {k: [] for k in libs}
        for _ in range(a.rounds):
            for k, lib in libs.items():
                env = dict(os.environ, RSSYNC_B200_LIB=os.path.abspath(lib))
                r = subprocess.run([sys.executable, os.path.abspath(pt.__file__), "--child", "--reps", str(a.reps)],
                                   env=env, capture_output=True, text=True, check=True)
                runs[k].append(json.loads(r.stdout.strip().splitlines()[-1]))
        digests = {k: sorted({x["digest"] for x in v}) for k, v in runs.items()}
        all_ms = {k: [m for x in v for m in x["ms"]] for k, v in runs.items()}
        res["no_mask_vs_base"] = {
            "case": "track_frames_ex_device, 64 frames at 2704 x 2028, selection and backward check",
            "call_ms": {k: pt._stats(v) for k, v in all_ms.items()},
            "ms_round_medians": {k: [float(np.median(x["ms"])) for x in v] for k, v in runs.items()},
            "bit_identical": digests["this"] == digests["base"] and len(digests["this"]) == 1, "digests": digests}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "prof_track_mask.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
