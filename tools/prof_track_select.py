"""Measure point selection and the forward-backward check of rssync_track_frames_ex_device on 64 frames of
rendered 2704 x 2028 luma planes (tests/render_reference.py).

  (a) per call of 64 frames, median and p10-p90 of a host clock around the call ending in a synchronise:
      track_frames on the 200-px grid, track_frames_ex with selection (defaults, fb_max = 0), and
      track_frames_ex with selection and the backward check (defaults, fb_max = 1 px);
  (b) per-kernel times of each from torch.profiler, in a separate pass;
  (c) with --base-lib (a build of the parent commit): track_frames on the grid through this build and
      through the base build, alternating in subprocesses over plain ctypes; the tracked positions, statuses
      and frame tables must be bit-identical.

The card's name, power limit and max SM clock are read in the same run.  Writes prof_track_select.json to
--out."""
from __future__ import annotations

import argparse
import hashlib
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
KERNELS = ("track_pyramid_kernel", "select_cells_kernel", "select_points_kernel", "select_prefix_kernel",
           "track_lk_kernel<false>", "track_lk_kernel<true>", "track_compact_kernel")


def gpu_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0),
            "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None}


def _clip():
    import render_reference as rr
    clip = rr.Clip(2704, 2028, 65, delay=0.037, seed=7)
    return clip, clip.render_all("cuda:0")


def _stats(ms):
    return {"median": float(np.median(ms)), "p10_p90": [float(np.percentile(ms, 10)), float(np.percentile(ms, 90))]}


def timing(reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    rsb = importlib.import_module("rs-sync_b200")
    clip, imgs = _clip()
    grid = rsb.grid_points(2704, 2028, 200)
    counts = np.full(64, grid.shape[0])
    pts = torch.from_numpy(np.tile(grid, (64, 1))).cuda()
    ids, ts, lens = clip.frame_ids(), clip.image_ts(), clip.lens()
    cases = {
        "track_frames_grid200": lambda p: p.track_frames(ids, counts, ts, pts, imgs, lens)[1],
        "track_frames_ex_select": lambda p: p.track_frames_ex(ids, ts, imgs, lens,
                                                              options=rsb.TrackOptions(fb_max=0.0)).status,
        "track_frames_ex_select_fb": lambda p: p.track_frames_ex(ids, ts, imgs, lens,
                                                                 options=rsb.TrackOptions(fb_max=1.0)).status,
    }
    out = {}
    for name, call in cases.items():
        ms = []
        for i in range(reps + 1):
            p = rsb.SyncProblem(seed=100)
            p.SetGyroQuaternions(clip.quats, clip.quats.shape[0], clip.gyro_rate, clip.gyro_t0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            st = call(p)
            torch.cuda.synchronize()
            if i:
                ms.append((time.perf_counter() - t0) * 1e3)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                call(p)
            torch.cuda.synchronize()
        kt = {}
        for e in prof.key_averages():
            for k in KERNELS:
                base, _, tmpl = k.partition("<")
                if base in e.key and (not tmpl or ("<" + tmpl) in e.key.replace(" ", "")):
                    kt[k] = kt.get(k, 0.0) + e.device_time_total / 1e3 / reps  # ms per call
        out[name] = {"frames_per_call": 64, "points": int(st.numel()),
                     "status_counts": {str(v): int((st == v).sum()) for v in (0, 1, 2)},
                     "call_ms": _stats(ms), "ms_per_frame_median": float(np.median(ms)) / 64,
                     "kernel_ms_per_call": kt}
    return out


def child(reps):
    """track_frames on the 200-px grid through RSSYNC_B200_LIB (plain ctypes: the base build lacks the new
    entry point)"""
    import ctypes as C
    import torch
    clip, imgs = _clip()
    rsb = importlib.import_module("rs-sync_b200")
    grid = rsb.grid_points(2704, 2028, 200)
    L = C.CDLL(os.environ["RSSYNC_B200_LIB"])
    P, dp, ip, sp = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_size_t)
    L.rssync_create.argtypes = [C.POINTER(P)]
    L.rssync_destroy.argtypes = [P]
    L.rssync_set_gyro_fixed.argtypes = [P, dp, C.c_size_t, C.c_double, C.c_double]
    L.rssync_track_frames_device.argtypes = [P, C.c_size_t, ip, sp, dp, P, P, C.c_size_t, C.c_int, C.c_int, dp, P,
                                             P, P, P]
    L.rssync_frame_table.argtypes = [P, C.c_void_p, C.c_size_t]
    n = 64 * grid.shape[0]
    pts = torch.from_numpy(np.tile(grid, (64, 1))).cuda()
    tracked = torch.empty((n, 2), dtype=torch.float64, device="cuda")
    status = torch.empty((n,), dtype=torch.uint8, device="cuda")
    ids = np.ascontiguousarray(clip.frame_ids(), dtype=np.int64)
    counts = np.full(64, grid.shape[0], dtype=np.uint64)
    ts = np.ascontiguousarray(clip.image_ts())
    lens = np.ascontiguousarray(clip.lens(), dtype=np.float64)
    quats = np.ascontiguousarray(clip.quats)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ms, digest = [], None
    for i in range(reps + 1):
        h = P()
        assert L.rssync_create(C.byref(h)) == 0
        assert L.rssync_set_gyro_fixed(h, quats.ctypes.data_as(dp), quats.shape[0], clip.gyro_rate, clip.gyro_t0) == 0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        assert L.rssync_track_frames_device(h, 64, ids.ctypes.data_as(ip), counts.ctypes.data_as(sp),
                                            ts.ctypes.data_as(dp), C.c_void_p(pts.data_ptr()),
                                            C.c_void_p(imgs.data_ptr()), imgs.stride(1), 2704, 2028,
                                            lens.ctypes.data_as(dp), None, C.c_void_p(tracked.data_ptr()),
                                            C.c_void_p(status.data_ptr()), stream) == 0
        torch.cuda.synchronize()
        if i:
            ms.append((time.perf_counter() - t0) * 1e3)
        nf = L.rssync_frame_table(h, None, 0)
        buf = C.create_string_buffer(32 * nf)
        L.rssync_frame_table(h, buf, nf)
        digest = hashlib.sha256(buf.raw + tracked.cpu().numpy().tobytes() + status.cpu().numpy().tobytes()).hexdigest()
        L.rssync_destroy(h)
    print(json.dumps({"ms": ms, "digest": digest}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--base-lib", default=None)
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        child(a.reps)
        return
    res = {"gpu": gpu_info(), "frames_2704x2028": timing(a.reps)}
    if a.base_lib:
        libs = {"this": os.path.join(ROOT, "rs-sync_b200", "lib", "librssync_b200.so"), "base": a.base_lib}
        runs = {k: [] for k in libs}
        for _ in range(a.rounds):
            for k, lib in libs.items():
                env = dict(os.environ, RSSYNC_B200_LIB=os.path.abspath(lib))
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--reps", str(a.reps)],
                                   env=env, capture_output=True, text=True, check=True)
                runs[k].append(json.loads(r.stdout.strip().splitlines()[-1]))
        digests = {k: sorted({x["digest"] for x in v}) for k, v in runs.items()}
        res["track_frames_grid200_vs_base"] = {
            "ms_median": {k: float(np.median([m for x in v for m in x["ms"]])) for k, v in runs.items()},
            "ms_round_medians": {k: [float(np.median(x["ms"])) for x in v] for k, v in runs.items()},
            "bit_identical": digests["this"] == digests["base"] and len(digests["this"]) == 1, "digests": digests}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "prof_track_select.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
