"""Windowed searches (SyncProblem.readout_search_windows / rotation_search_windows) against the loop a caller
writes without them -- one single-window search per window, with the same call numbers -- on the C2 shape
(3300 frames x 200 pixel pairs or rays, its 1 kHz gyro) with PreSync's delay grid of C2 (D = 200):

  * readout: 12 readouts x W = 10 windows of 60 frames, from pixels;
  * rotation: 11 rotations about x (0-50 degrees) x the same windows;
  * drift: the readout search on C4s (C4's 30-minute trace with the delay drifting from -45 to -40 ms,
    only the frames of its sync windows tracked), one 60-frame window at each of driver.syncpoint_list's
    positions (every 1000 frames: 108 windows), a delay grid covering the drift;
  * the GPU's name, power limit and max SM clock, read in the same run.

Every windowed call ends in a device synchronise; medians over --reps repetitions with p10 / p90, the two
forms alternating.  The arena fits the L2 and is not flushed between calls.  The windowed (cost, delay)
arrays are checked bit for bit against the loop's.

With --base-lib LIB the single-window searches (readout_search over 11 readouts and rotation_search over
11 rotations on the whole C2 clip) are also timed for this build (--lib, default the package's library)
and LIB, alternating in subprocesses, --rounds rounds of --reps each, through a minimal ctypes binding of
the entry points both builds have; their results are compared bit for bit.  Needs a CUDA GPU and fails
without one.  Prints JSON; with --out DIR also writes DIR/prof_search_windows.json.

    python tools/prof_search_windows.py [--out DIR] [--reps 10] [--base-lib LIB] [--rounds 3]
"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_READOUTS, N_ROT, W, WINDOW = 12, 11, 10, 60


def gpu_info(device=0):
    import torch
    q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(device),
            "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None}


def timed(forms, reps):
    """{name: fn} alternating, the first round a warm-up -> ({name: ms list}, {name: last result})"""
    import torch
    t = {k: [] for k in forms}
    res = {}
    for i in range(reps + 1):
        for k, fn in forms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res[k] = fn()
            torch.cuda.synchronize()
            if i >= 1:
                t[k].append((time.perf_counter() - t0) * 1e3)
    return t, res


def summary(t):
    return {"ms_median": {k: float(np.median(v)) for k, v in t.items()},
            "ms_p10_p90": {k: [float(np.percentile(v, 10)), float(np.percentile(v, 90))] for k, v in t.items()}}


def same(a, b):
    return all(np.array_equal(np.asarray(x), np.asarray(y)) for x, y in zip(a, b))


def scene(pkg, synth, name):
    w = synth.make_workload(name, procs=min(16, os.cpu_count() or 1))
    ts = w.gyro_t0 + np.arange(w.quats.shape[0]) / w.gyro_rate
    return w, ts


def pixels_problem(pkg, synth, w):
    p = pkg.SyncProblem(seed=100)
    p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
    p.set_track_pixels(w.frame_ids, np.full(w.n_frames, w.n_rays), w.frame_ids / w.fps, (w.frame_ids + 1) / w.fps,
                       w.px_a.reshape(-1), w.px_b.reshape(-1), (float(synth.READOUT),) + tuple(synth.LENS[1:]),
                       synth.HEIGHT)
    p.flush()
    return p


def readout_case(pkg, p, readouts, fb, fe, initial, step, radius, reps):
    n = len(readouts)
    calls = np.arange(n * len(fb), dtype=np.uint64) + 50

    def windowed():
        return p.readout_search_windows(readouts, initial, fb, fe, step, radius, call_nos=calls)

    def loop():
        c, d = np.empty((n, len(fb))), np.empty((n, len(fb)))
        for k in range(len(fb)):
            c[:, k], d[:, k] = p.readout_search(readouts, initial, int(fb[k]), int(fe[k]), step, radius,
                                                call_nos=calls[k::len(fb)])
        return c, d

    t, res = timed({"windowed": windowed, "loop": loop}, reps)
    out = summary(t)
    out["results_bit_identical"] = bool(same(res["windowed"], res["loop"]))
    out["speedup"] = out["ms_median"]["loop"] / out["ms_median"]["windowed"]
    return out


def child(path, reps):
    """the single-window searches on the saved C2 scene through the library RSSYNC_B200_LIB names"""
    import torch
    pkg = importlib.import_module("rs-sync_b200")
    d = dict(np.load(path))
    L = C.CDLL(os.environ["RSSYNC_B200_LIB"])
    P, dp = C.c_void_p, C.POINTER(C.c_double)
    i64p, u64p = C.POINTER(C.c_int64), C.POINTER(C.c_uint64)
    L.rssync_create.argtypes = [C.POINTER(P)]
    L.rssync_destroy.argtypes = [P]
    L.rssync_flush.argtypes = [P]
    L.rssync_set_gyro_fixed.argtypes = [P, dp, C.c_size_t, C.c_double, C.c_double]
    L.rssync_set_track_pixels.argtypes = [P, C.c_size_t, i64p, C.POINTER(C.c_size_t), dp, dp, dp, dp,
                                          C.POINTER(pkg.Lens), C.c_double]
    L.rssync_readout_search.argtypes = [P, dp, C.c_int, C.c_double, C.c_int64, C.c_int64, C.c_double, C.c_double,
                                        u64p, dp, dp, dp]
    L.rssync_rotation_search.argtypes = [P, dp, dp, C.c_size_t, dp, C.c_int, C.c_double, C.c_int64, C.c_int64,
                                         C.c_double, C.c_double, u64p, dp, dp, dp]
    ptr = lambda a: a.ctypes.data_as(dp)
    h = P()
    assert L.rssync_create(C.byref(h)) == 0
    assert L.rssync_set_gyro_fixed(h, ptr(d["quats"]), d["quats"].shape[0], float(d["gyro_rate"]),
                                   float(d["gyro_t0"])) == 0
    ids = d["frame_ids"].astype(np.int64)
    counts = np.full(ids.size, d["px_a"].shape[1], dtype=np.uint64)
    lens = pkg.Lens(*[float(x) for x in d["lens"]])
    pa, pb = np.ascontiguousarray(d["px_a"].reshape(-1)), np.ascontiguousarray(d["px_b"].reshape(-1))
    ta, tb = np.ascontiguousarray(d["ts_a"]), np.ascontiguousarray(d["ts_b"])
    assert L.rssync_set_track_pixels(h, ids.size, ids.ctypes.data_as(i64p), counts.ctypes.data_as(C.POINTER(C.c_size_t)),
                                     ptr(ta), ptr(tb), ptr(pa), ptr(pb), C.byref(lens), float(d["height"])) == 0
    assert L.rssync_flush(h) == 0
    fb, fe = int(ids[0]), int(ids[-1]) + 1
    initial, step, radius = 0.0, float(d["step"]), float(d["radius"])
    readouts, rots = d["readouts"], np.ascontiguousarray(d["rots"])
    calls = np.arange(11, dtype=np.uint64) + 50
    cu = calls.ctypes.data_as(u64p)
    rc_, rd = np.empty(len(readouts)), np.empty(len(readouts))
    oc, od = np.empty(len(rots)), np.empty(len(rots))
    ts, om = np.ascontiguousarray(d["ts"]), np.ascontiguousarray(d["omega"])

    def readout():
        assert L.rssync_readout_search(h, ptr(readouts), len(readouts), initial, fb, fe, step, radius, cu, ptr(rc_),
                                       ptr(rd), None) == 0

    def rotation():
        assert L.rssync_rotation_search(h, ptr(ts), ptr(om), ts.shape[0], ptr(rots), len(rots), initial, fb, fe,
                                        step, radius, cu, ptr(oc), ptr(od), None) == 0

    t, _ = timed({"readout_search": readout, "rotation_search": rotation}, reps)
    L.rssync_destroy(h)
    print(json.dumps({"ms": t, "results": [rc_.tolist(), rd.tolist(), oc.tolist(), od.tolist()]}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for prof_search_windows.json (default: print only)")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3, help="alternating rounds per library (--base-lib)")
    ap.add_argument("--lib", default=None, help="this build (default: the package's library)")
    ap.add_argument("--base-lib", default=None, help="the build to compare the single-window searches against")
    ap.add_argument("--child", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:
        return child(args.child, args.reps)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("prof_search_windows: no CUDA device (this measurement has no CPU form)")
    pkg = importlib.import_module("rs-sync_b200")
    synth = importlib.import_module("rs-sync_b200.synth")
    driver = importlib.import_module("rs-sync_b200.driver")
    out = {"gpu": gpu_info(), "reps": args.reps}
    w, ts = scene(pkg, synth, "C2")
    initial, step, radius = 0.0, w.presync_step, w.presync_radius
    D = int(pkg.presync_delays(initial, step, radius).shape[0])
    f0 = int(w.frame_ids[0])
    stride = (w.n_frames - WINDOW) // (W - 1)
    fb = f0 + stride * np.arange(W, dtype=np.int64)
    fe = fb + WINDOW
    out["shape"] = {"frames": w.n_frames, "pairs_per_frame": w.n_rays, "windows": W, "window_frames": WINDOW,
                    "delays": D, "readouts": N_READOUTS, "rotations": N_ROT}
    # ---- readout, C2 from pixels -----------------------------------------------------------------------
    p = pixels_problem(pkg, synth, w)
    readouts = np.linspace(0.0, 0.022, N_READOUTS)
    out["readout"] = readout_case(pkg, p, readouts, fb, fe, initial, step, radius, args.reps)
    p.close()
    # ---- rotation, C2 ----------------------------------------------------------------------------------
    g = pkg.SyncProblem(seed=100).load(w, bulk=True)
    g.flush()
    rots = pkg.rotations_about("x", np.deg2rad(np.linspace(0.0, 50.0, N_ROT)))
    calls = np.arange(N_ROT * W, dtype=np.uint64) + 50

    def windowed():
        return g.rotation_search_windows(ts, w.omega, rots, initial, fb, fe, step, radius, call_nos=calls)

    def loop():
        c, d = np.empty((N_ROT, W)), np.empty((N_ROT, W))
        for k in range(W):
            c[:, k], d[:, k] = g.rotation_search(ts, w.omega, rots, initial, int(fb[k]), int(fe[k]), step, radius,
                                                 call_nos=calls[k::W])
        return c, d

    t, res = timed({"windowed": windowed, "loop": loop}, args.reps)
    out["rotation"] = summary(t)
    out["rotation"]["results_bit_identical"] = bool(same(res["windowed"], res["loop"]))
    out["rotation"]["speedup"] = out["rotation"]["ms_median"]["loop"] / out["rotation"]["ms_median"]["windowed"]
    g.close()
    # ---- a drifting C4-shaped clip, windows at the syncpoints ---------------------------------------------
    w4, _ = scene(pkg, synth, "C4s")  # C4's 30-minute trace, only the frames of its sync windows tracked
    cfg = {"input": {"frame_range": [0, 108000]},
           "params": {"syncpoints_format": "auto", "sync_window": WINDOW, "syncpoint_distance": 1000}}
    pos = np.array(driver.syncpoint_list(cfg), dtype=np.int64)
    p4 = pixels_problem(pkg, synth, w4)
    i4, s4, r4 = -0.0425, w4.presync_step, max(w4.presync_radius, 0.02)
    out["drift"] = readout_case(pkg, p4, readouts, pos, pos + WINDOW, i4, s4, r4, args.reps)
    out["drift"]["shape"] = {"frames": w4.n_frames, "pairs_per_frame": w4.n_rays, "windows": int(pos.size),
                             "window_frames": WINDOW, "initial": i4, "radius": r4,
                             "delays": int(pkg.presync_delays(i4, s4, r4).shape[0])}
    p4.close()
    # ---- the single-window searches against another build ------------------------------------------------
    if args.base_lib:
        libs = {"this": args.lib or pkg.LIB_PATH, "base": args.base_lib}
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "c2.npz")
            np.savez(path, quats=w.quats, gyro_rate=w.gyro_rate, gyro_t0=w.gyro_t0, frame_ids=w.frame_ids,
                     px_a=w.px_a, px_b=w.px_b, ts_a=w.frame_ids / w.fps, ts_b=(w.frame_ids + 1) / w.fps,
                     lens=np.array((float(synth.READOUT),) + tuple(synth.LENS[1:])), height=synth.HEIGHT,
                     step=step, radius=radius, readouts=np.linspace(0.0, 0.02, 11), rots=rots, ts=ts,
                     omega=w.omega)
            runs = {k: [] for k in libs}
            for _ in range(args.rounds):
                for k, lib in libs.items():
                    env = dict(os.environ, RSSYNC_B200_LIB=os.path.abspath(lib))
                    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", path, "--reps",
                                        str(args.reps)], env=env, capture_output=True, text=True, check=True)
                    runs[k].append(json.loads(r.stdout.strip().splitlines()[-1]))
        cmp = {"rounds": args.rounds, "reps_per_round": args.reps}
        for k, rs in runs.items():
            cmp[k] = {}
            for form in ("readout_search", "rotation_search"):
                allv = [x for r in rs for x in r["ms"][form]]
                cmp[k][form] = {"ms_median": float(np.median(allv)),
                                "round_medians": [float(np.median(r["ms"][form])) for r in rs]}
        cmp["results_bit_identical"] = all(r["results"] == runs["this"][0]["results"] for rs in runs.values()
                                           for r in rs)
        out["single_window_vs_base"] = cmp
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "prof_search_windows.json"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
