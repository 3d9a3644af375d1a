"""Measure rssync_track_frames_device on rendered 2704 x 2028 luma planes (tests/render_reference.py).

  (a) time per frame of track_frames in batches of 64 frames, for the reference's 200-px grid and for 500
      points per frame: a host clock around each call ending in a synchronise, and per-kernel times
      (track_pyramid_kernel, track_lk_kernel, track_compact_kernel) from torch.profiler in a separate pass;
  (b) the pyramid kernel's bytes, computed from the shapes, as a share of 7.7 TB/s;
  (c) for context, on the same host: cv2.calcOpticalFlowPyrLK, and cv2.DISOpticalFlow (medium) plus grid
      sampling, per frame, with cv2's thread count;
  (d) set_track_pixels_device + a PreSync grid on C2's pixel pairs through this build and through --base-lib
      (e.g. a build of the parent commit), alternating in subprocesses; results must be bit-identical.

The card's name, power limit and max SM clock are read in the same run.  Writes prof_track.json to --out."""
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
KERNELS = ("track_pyramid_kernel", "track_lk_kernel", "track_compact_kernel")


def gpu_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0),
            "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None}


def pyramid_bytes(w, h, levels, images):
    """level 0 read as uint8, levels >= 1 written and (but the last) read as float32, per image"""
    b, lw, lh = 0, w, h
    for lvl in range(levels - 1):
        nw, nh = (lw + 1) // 2, (lh + 1) // 2
        b += (lw * lh * (1 if lvl == 0 else 4)) + 4 * nw * nh
        lw, lh = nw, nh
    return b * images


def track_timing(reps):
    import torch
    rsb = importlib.import_module("rs-sync_b200")
    import render_reference as rr
    clip = rr.Clip(2704, 2028, 65, delay=0.037, seed=7)
    imgs = clip.render_all("cuda:0")
    rng = np.random.default_rng(1)
    grid = rsb.grid_points(2704, 2028, 200)
    rand500 = np.stack([rng.uniform(20, 2683, 500), rng.uniform(20, 2007, 500)], axis=-1)
    out = {}
    for name, q in (("grid200", grid), ("points500", rand500)):
        counts = np.full(64, q.shape[0])
        pts = torch.from_numpy(np.tile(q, (64, 1))).cuda()
        ids, ts = clip.frame_ids(), clip.image_ts()

        def call(p):
            return p.track_frames(ids, counts, ts, pts, imgs, clip.lens())

        ms = []
        for i in range(reps + 1):
            p = rsb.SyncProblem(seed=100)
            p.SetGyroQuaternions(clip.quats, clip.quats.shape[0], clip.gyro_rate, clip.gyro_t0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, st = call(p)
            torch.cuda.synchronize()
            if i:
                ms.append((time.perf_counter() - t0) * 1e3)
        kept = float(st.float().mean())
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                call(p)
            torch.cuda.synchronize()
        kt = {k: 0.0 for k in KERNELS}
        for e in prof.key_averages():
            for k in KERNELS:
                if k in e.key:
                    kt[k] += e.device_time_total / 1e3 / reps  # ms per call
        pb = pyramid_bytes(2704, 2028, 3, 65)
        out[name] = {"points_per_frame": int(q.shape[0]), "frames_per_call": 64, "kept_fraction": kept,
                     "call_ms_median": float(np.median(ms)), "call_ms_p10_p90": [float(np.percentile(ms, 10)),
                                                                                 float(np.percentile(ms, 90))],
                     "ms_per_frame": float(np.median(ms)) / 64, "kernel_ms_per_call": kt,
                     "pyramid_bytes_per_call": pb,
                     "pyramid_share_of_7.7TBps": (pb / (kt["track_pyramid_kernel"] * 1e-3)) / 7.7e12
                     if kt["track_pyramid_kernel"] else None}
    # (c) host cv2 for context
    import cv2
    host = imgs[:9].cpu().numpy()
    crit = (cv2.TERM_CRITERIA_COUNT | cv2.TERM_CRITERIA_EPS, 30, 0.01)
    t0 = time.perf_counter()
    for j in range(8):
        cv2.calcOpticalFlowPyrLK(host[j], host[j + 1], grid.astype(np.float32).reshape(-1, 1, 2), None,
                                 winSize=(21, 21), maxLevel=2, criteria=crit)
    lk = (time.perf_counter() - t0) / 8 * 1e3
    dis = cv2.DISOpticalFlow_create(cv2.DISOPTICAL_FLOW_PRESET_MEDIUM)
    t0 = time.perf_counter()
    for j in range(8):
        f = dis.calc(host[j], host[j + 1], None)
        _ = f[np.rint(grid[:, 1]).astype(int), np.rint(grid[:, 0]).astype(int)]
    dm = (time.perf_counter() - t0) / 8 * 1e3
    out["host_context"] = {"cv2_threads": cv2.getNumThreads(), "cpu_count": os.cpu_count(),
                           "cv2_calcOpticalFlowPyrLK_grid200_ms_per_frame": lk,
                           "cv2_DIS_medium_plus_grid_ms_per_frame": dm}
    return out


def child(path, reps):
    """set_track_pixels_device and a PreSync grid on the saved C2 pixels through RSSYNC_B200_LIB"""
    import ctypes as C
    import torch
    L = C.CDLL(os.environ["RSSYNC_B200_LIB"])
    P, dp, ip, sp = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_size_t)
    L.rssync_create.argtypes = [C.POINTER(P)]
    L.rssync_destroy.argtypes = [P]
    L.rssync_set_gyro_fixed.argtypes = [P, dp, C.c_size_t, C.c_double, C.c_double]
    L.rssync_set_track_pixels_device.argtypes = [P, C.c_size_t, ip, sp, dp, dp, P, P, dp, C.c_double, P]
    L.rssync_presync_grid.argtypes = [P, C.c_int64, C.c_int64, dp, C.c_int, C.c_int, C.c_uint64, C.c_uint64, dp,
                                      C.POINTER(C.c_uint)]
    L.rssync_frame_table.argtypes = [P, C.c_void_p, C.c_size_t]
    d = {k: np.ascontiguousarray(v) for k, v in np.load(path).items()}
    ptr = lambda a: a.ctypes.data_as(dp)  # noqa: E731
    F, N = d["px_a"].shape[:2]
    ids = d["frame_ids"].astype(np.int64)
    counts = np.full(F, N, dtype=np.uint64)
    fta, ftb = ids / float(d["fps"]), (ids + 1) / float(d["fps"])
    pa, pb = torch.from_numpy(d["px_a"]).cuda(), torch.from_numpy(d["px_b"]).cuda()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    delays = np.ascontiguousarray(d["delays"])
    curve = np.empty(delays.shape[0])
    flags = C.c_uint()
    ms, digest = [], None
    for i in range(reps + 1):
        h = P()
        assert L.rssync_create(C.byref(h)) == 0
        assert L.rssync_set_gyro_fixed(h, ptr(d["quats"]), d["quats"].shape[0], float(d["gyro_rate"]),
                                       float(d["gyro_t0"])) == 0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        assert L.rssync_set_track_pixels_device(h, F, ids.ctypes.data_as(ip), counts.ctypes.data_as(sp), ptr(fta),
                                                ptr(ftb), C.c_void_p(pa.data_ptr()), C.c_void_p(pb.data_ptr()),
                                                ptr(d["lens"]), float(d["rows"]), stream) == 0
        assert L.rssync_presync_grid(h, int(ids[0]), int(ids[-1]) + 1, ptr(delays), delays.shape[0], 1, 7, 0,
                                     ptr(curve), C.byref(flags)) == 0
        torch.cuda.synchronize()
        if i:
            ms.append((time.perf_counter() - t0) * 1e3)
        n = L.rssync_frame_table(h, None, 0)
        buf = C.create_string_buffer(32 * n)
        L.rssync_frame_table(h, buf, n)
        digest = hashlib.sha256(buf.raw + curve.tobytes() + np.uint32(flags.value).tobytes()).hexdigest()
        L.rssync_destroy(h)
    print(json.dumps({"ms": ms, "digest": digest}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--base-lib", default=None)
    ap.add_argument("--child", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        child(a.child, a.reps)
        return
    res = {"gpu": gpu_info(), "track_frames_2704x2028": track_timing(a.reps)}
    if a.base_lib:
        import tempfile
        synth = importlib.import_module("rs-sync_b200.synth")
        rsb = importlib.import_module("rs-sync_b200")
        w = synth.make_workload("C2", procs=os.cpu_count() or 1)
        tmp = tempfile.mkdtemp()
        path = os.path.join(tmp, "c2.npz")
        np.savez(path, px_a=w.px_a, px_b=w.px_b, frame_ids=w.frame_ids, fps=w.fps, quats=w.quats,
                 gyro_rate=w.gyro_rate, gyro_t0=w.gyro_t0, lens=np.array(synth.LENS), rows=float(synth.HEIGHT),
                 delays=rsb.presync_delays(0.0, w.presync_step, w.presync_radius))
        libs = {"this": os.path.join(ROOT, "rs-sync_b200", "lib", "librssync_b200.so"), "base": a.base_lib}
        runs = {k: [] for k in libs}
        for _ in range(a.rounds):
            for k, lib in libs.items():
                env = dict(os.environ, RSSYNC_B200_LIB=os.path.abspath(lib))
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", path, "--reps", str(a.reps)],
                                   env=env, capture_output=True, text=True, check=True)
                runs[k].append(json.loads(r.stdout.strip().splitlines()[-1]))
        digests = {k: sorted({x["digest"] for x in v}) for k, v in runs.items()}
        res["pixels_device_plus_c2_presync_vs_base"] = {
            "ms_median": {k: float(np.median([m for x in v for m in x["ms"]])) for k, v in runs.items()},
            "ms_round_medians": {k: [float(np.median(x["ms"])) for x in v] for k, v in runs.items()},
            "bit_identical": digests["this"] == digests["base"] and len(digests["this"]) == 1, "digests": digests}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "prof_track.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
