"""Measure tracking on 16-bit luma planes (rssync_track_frames16_device) against the 8-bit path, on 64 frames of
rendered luma planes (tests/render_reference.py) at 2704 x 2028 and 3840 x 2160, with selection and the
backward check on (TrackOptions defaults: 128-px cells, block 5, 512 points, fb_max 1 px).

  (a) per call of 64 frames, median and p10-p90 of a host clock around the call ending in a synchronise, the
      three cases alternating: the 8-bit path on P, the 16-bit path on P010 samples P << 8 (shift 8), and the
      workaround a caller of the 8-bit path needs today: a narrowing pass (the high byte of every P010 sample,
      one copy kernel) and then the 8-bit path.  The 16-bit outputs must equal the 8-bit ones bit for bit;
  (b) per-kernel times of each case from torch.profiler, in a separate pass;
  (c) the level-0 plane bytes each case reads (and writes, for the narrowing pass), from the shapes;
  (d) with --base-lib (a build of the parent commit): the 8-bit path at 2704 x 2028 through this build and
      through the base build, alternating in subprocesses over plain ctypes; the outputs and frame tables must
      be bit-identical.

The card's name, power limit and max SM clock are read in the same run.  Writes prof_track16.json to --out."""
from __future__ import annotations

import argparse
import ctypes as C
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
           "track_lk_kernel", "track_compact_kernel")
SIZES = ((2704, 2028), (3840, 2160))


def gpu_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0),
            "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None}


def _clip(w, h):
    import render_reference as rr
    clip = rr.Clip(w, h, 65, delay=0.037, seed=7)
    return clip, clip.render_all("cuda:0")


def _stats(ms):
    return {"median": float(np.median(ms)), "p10_p90": [float(np.percentile(ms, 10)), float(np.percentile(ms, 90))]}


def timing(w, h, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    rsb = importlib.import_module("rs-sync_b200")
    clip, imgs = _clip(w, h)
    p010 = torch.from_numpy(imgs.cpu().numpy().astype(np.uint16) << 8).cuda()
    ids, ts, lens = clip.frame_ids(), clip.image_ts(), clip.lens()
    opt = rsb.TrackOptions()

    def problem():
        p = rsb.SyncProblem(seed=100)
        p.SetGyroQuaternions(clip.quats, clip.quats.shape[0], clip.gyro_rate, clip.gyro_t0)
        return p

    def narrow(x):
        return x.view(torch.uint8)[:, :, 1::2].contiguous()  # the high byte (little-endian) of each sample

    cases = {
        "8bit": lambda p: p.track_frames_ex(ids, ts, imgs, lens, options=opt),
        "16bit_shift8": lambda p: p.track_frames_ex(ids, ts, p010, lens, options=opt, shift=8),
        "narrow_then_8bit": lambda p: p.track_frames_ex(ids, ts, narrow(p010), lens, options=opt),
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
    ref = res["8bit"]
    identical = {k: all(getattr(r, f).cpu().numpy().tobytes() == getattr(ref, f).cpu().numpy().tobytes()
                        for f in ("points", "tracked", "status", "fb_error")) and
                 np.array_equal(r.counts, ref.counts) for k, r in res.items()}
    out = {}
    n_img, px = 65, w * h
    level0 = {"8bit": {"read": n_img * px}, "16bit_shift8": {"read": 2 * n_img * px},
              "narrow_then_8bit": {"narrow_read": 2 * n_img * px, "narrow_write": n_img * px, "read": n_img * px}}
    for name, call in cases.items():
        p = problem()
        call(p)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                call(problem())
            torch.cuda.synchronize()
        kt = {}
        for e in prof.key_averages():
            k = next((k for k in KERNELS if k in e.key), None)
            key = k + ("<uint16>" if "unsigned short" in e.key else "") if k else None
            if key is None and ("copy" in e.key.lower() or "elementwise" in e.key.lower()):
                key = "torch: " + e.key[:80]
            if key:
                kt[key] = kt.get(key, 0.0) + e.device_time_total / 1e3 / reps  # ms per call
        st = res[name].status
        out[name] = {"frames_per_call": 64, "points": int(st.numel()),
                     "status_counts": {str(v): int((st == v).sum()) for v in (0, 1, 2)},
                     "call_ms": _stats(ms[name]), "kernel_ms_per_call": kt, "level0_bytes": level0[name],
                     "outputs_equal_8bit": identical[name]}
    return out


class _Opt(C.Structure):
    _fields_ = [("cell", C.c_int), ("block", C.c_int), ("quality", C.c_double), ("max_points", C.c_int),
                ("fb_max", C.c_double)]


def child(reps):
    """the 8-bit path (rssync_track_frames_ex_device, selection and the backward check) at 2704 x 2028 through
    RSSYNC_B200_LIB over plain ctypes"""
    import torch
    clip, imgs = _clip(2704, 2028)
    L = C.CDLL(os.environ["RSSYNC_B200_LIB"])
    P, dp, ip, sp = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_size_t)
    L.rssync_create.argtypes = [C.POINTER(P)]
    L.rssync_destroy.argtypes = [P]
    L.rssync_set_gyro_fixed.argtypes = [P, dp, C.c_size_t, C.c_double, C.c_double]
    L.rssync_track_frames_ex_device.argtypes = [P, C.c_size_t, ip, sp, dp, P, P, C.c_size_t, C.c_int, C.c_int, dp,
                                                P, C.POINTER(_Opt), P, sp, P, P, P, P]
    L.rssync_frame_table.argtypes = [P, C.c_void_p, C.c_size_t]
    opt = _Opt(128, 5, 0.01, 512, 1.0)
    n = 64 * 512
    bufs = [torch.empty(s, dtype=d, device="cuda") for s, d in (((n, 2), torch.float64), ((n, 2), torch.float64),
                                                               ((n,), torch.uint8), ((n,), torch.float64))]
    counts = np.zeros(64, dtype=np.uint64)
    ids = np.ascontiguousarray(clip.frame_ids(), dtype=np.int64)
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
        assert L.rssync_track_frames_ex_device(h, 64, ids.ctypes.data_as(ip), None, ts.ctypes.data_as(dp), None,
                                               C.c_void_p(imgs.data_ptr()), imgs.stride(1), 2704, 2028,
                                               lens.ctypes.data_as(dp), None, C.byref(opt),
                                               *[C.c_void_p(b.data_ptr()) for b in bufs[:1]],
                                               counts.ctypes.data_as(sp),
                                               *[C.c_void_p(b.data_ptr()) for b in bufs[1:]], stream) == 0
        torch.cuda.synchronize()
        if i:
            ms.append((time.perf_counter() - t0) * 1e3)
        nf = L.rssync_frame_table(h, None, 0)
        buf = C.create_string_buffer(32 * nf)
        L.rssync_frame_table(h, buf, nf)
        k = int(counts.sum())
        digest = hashlib.sha256(buf.raw + counts.tobytes() + b"".join(b[:k].cpu().numpy().tobytes()
                                                                      for b in bufs)).hexdigest()
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
    res = {"gpu": gpu_info()}
    for w, h in SIZES:
        res[f"frames_{w}x{h}"] = timing(w, h, a.reps)
    res["8bit_vs_base"] = "not measured (no --base-lib)"
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
        res["8bit_vs_base"] = {
            "case": "track_frames_ex_device, 64 frames at 2704 x 2028, selection and backward check",
            "ms_median": {k: float(np.median([m for x in v for m in x["ms"]])) for k, v in runs.items()},
            "ms_round_medians": {k: [float(np.median(x["ms"])) for x in v] for k, v in runs.items()},
            "bit_identical": digests["this"] == digests["base"] and len(digests["this"]) == 1, "digests": digests}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "prof_track16.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
