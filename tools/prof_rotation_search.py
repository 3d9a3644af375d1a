"""Rotation search (SyncProblem.rotation_search, rssync_rotation_search) against the loop a caller writes
without it, and the orientation search (C5) on two builds of the library.

  (a) C2 shape (3300 frames x 200 rays, its 1 kHz gyro), 11 candidate rotations about x (0 .. 50 degrees),
      PreSync's delay grid of C2 (step 2 ms, radius 0.2 s: D = 200 offsets):
        * search: one rotation_search call over the 11 matrices (it ends in a device synchronise);
        * loop: per matrix integrate_gyro(rotation=) on the host, the variable-rate SetGyroQuaternions and
          PreSync on one problem -- what a caller does without the search;
        * search without frames in range: the gyro pipeline alone (integration, resampling, records).
      Medians over --reps repetitions, the forms alternating; results checked bit for bit at the same RNG
      call numbers.
  (b) C5: the 48-string orientation search on C2, timed in subprocesses that load the library named by
      --lib and by --base-lib (e.g. a build of the parent commit into another directory) through
      RSSYNC_B200_LIB, alternating, --rounds rounds of --reps searches each.  The two builds' (cost, delay)
      pairs are compared bit for bit.
  (c) the GPU's name, power limit and max SM clock, read in the same run.

Needs a CUDA GPU and fails without one.  Prints the results as JSON; with --out DIR also writes them to
DIR/prof_rotation_search.json.

    python tools/prof_rotation_search.py [--out DIR] [--reps 10] [--base-lib PATH] [--lib PATH] [--rounds 3]
"""
import argparse
import importlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0),
            "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None}


def c5_child(path, reps):
    """the 48-string orientation search on the saved C2 scene, through a minimal ctypes binding of the library
    RSSYNC_B200_LIB names (the entry points every build has, so a build of an older commit loads too)"""
    import ctypes as C
    import torch
    synth = importlib.import_module("rs-sync_b200.synth")
    lib_path = os.environ["RSSYNC_B200_LIB"]
    L = C.CDLL(lib_path)
    P, dp = C.c_void_p, C.POINTER(C.c_double)
    L.rssync_create.argtypes = [C.POINTER(P)]
    L.rssync_destroy.argtypes = [P]
    L.rssync_set_rng.argtypes = [P, C.c_uint64, C.c_uint64]
    L.rssync_set_gyro_fixed.argtypes = [P, dp, C.c_size_t, C.c_double, C.c_double]
    L.rssync_set_track_batch.argtypes = [P, C.c_size_t, C.POINTER(C.c_int64), C.POINTER(C.c_size_t), dp, dp, dp, dp]
    L.rssync_flush.argtypes = [P]
    L.rssync_orientation_search_ex.argtypes = [P, dp, dp, C.c_size_t, C.POINTER(C.c_char_p), C.c_int, C.c_double,
                                               C.c_int64, C.c_int64, C.c_double, C.c_double, C.POINTER(C.c_uint64),
                                               dp, dp]
    d = {k: np.ascontiguousarray(v) for k, v in np.load(path).items()}
    ptr = lambda a: a.ctypes.data_as(dp)
    h = P()
    assert L.rssync_create(C.byref(h)) == 0
    assert L.rssync_set_gyro_fixed(h, ptr(d["quats"]), d["quats"].shape[0], float(d["gyro_rate"]),
                                   float(d["gyro_t0"])) == 0
    F, N = d["ts_a"].shape
    ids = d["frame_ids"].astype(np.int64)
    counts = np.full(F, N, dtype=np.uint64)
    assert L.rssync_set_track_batch(h, F, ids.ctypes.data_as(C.POINTER(C.c_int64)),
                                    counts.ctypes.data_as(C.POINTER(C.c_size_t)), ptr(d["ts_a"]), ptr(d["ts_b"]),
                                    ptr(d["rays_a"]), ptr(d["rays_b"])) == 0
    assert L.rssync_flush(h) == 0
    fb, fe = int(ids[0]), int(ids[-1]) + 1
    n = len(synth.ORIENTATIONS)
    names = (C.c_char_p * n)(*[o.encode() for o in synth.ORIENTATIONS])
    cost, delay = np.empty(n), np.empty(n)
    ms = []
    for i in range(reps + 1):
        L.rssync_set_rng(h, 100, 0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rc = L.rssync_orientation_search_ex(h, ptr(d["ts"]), ptr(d["omega"]), d["ts"].shape[0], names, n, 0.0, fb, fe,
                                            float(d["step"]), float(d["radius"]), None, ptr(cost), ptr(delay))
        torch.cuda.synchronize()
        assert rc == 0, rc
        if i:
            ms.append((time.perf_counter() - t0) * 1e3)
    L.rssync_destroy(h)
    print(json.dumps({"lib": lib_path, "ms": ms, "cost": cost.tolist(), "delay": delay.tolist()}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for prof_rotation_search.json (default: print only)")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3, help="C5: alternating rounds per library")
    ap.add_argument("--lib", default=None, help="C5: this build (default: the package's library)")
    ap.add_argument("--base-lib", default=None, help="C5: the build to compare against (default: none)")
    ap.add_argument("--c5-child", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.c5_child:
        return c5_child(args.c5_child, args.reps)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("prof_rotation_search: no CUDA device (this measurement has no CPU form)")
    pkg = importlib.import_module("rs-sync_b200")
    synth = importlib.import_module("rs-sync_b200.synth")
    out = {"gpu": gpu_info()}
    w = synth.make_workload("C2", procs=min(16, os.cpu_count() or 1))
    ts = w.gyro_t0 + np.arange(w.quats.shape[0]) / w.gyro_rate
    ts_us = (ts * 1000000).astype(np.int64)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    initial, step, radius = 0.0, w.presync_step, w.presync_radius
    D = pkg.presync_delays(initial, step, radius).shape[0]
    angles = np.deg2rad(np.linspace(0.0, 50.0, 11))
    rots = pkg.rotations_about("x", angles)
    calls = np.arange(len(rots), dtype=np.uint64) + 50
    # ---- (a) ------------------------------------------------------------------------------------------
    p = pkg.SyncProblem(seed=100).load(w, bulk=True)
    p.flush()
    loop = pkg.SyncProblem(seed=100).load(w, bulk=True)
    loop.flush()

    def run_search():
        return p.rotation_search(ts, w.omega, rots, initial, fb, fe, step, radius, call_nos=calls)

    def run_loop():
        res = []
        for m, c in zip(rots, calls):
            loop.SetGyroQuaternions(ts_us, pkg.integrate_gyro(ts, w.omega, rotation=m), len(ts_us))
            loop.set_rng(100, int(c))
            res.append(loop.PreSync(initial, fb, fe, step, radius))
        return res

    def run_gyro_only():
        return p.rotation_search(ts, w.omega, rots, initial, 10 ** 7, 10 ** 7 + 1, step, radius, call_nos=calls)

    forms = {"search": run_search, "loop": run_loop, "search_no_frames": run_gyro_only}
    t = {k: [] for k in forms}
    results = {}
    for i in range(args.reps + 1):
        for k, fn in forms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            results[k] = fn()
            torch.cuda.synchronize()
            if i >= 1:  # the first round warms every shape up
                t[k].append((time.perf_counter() - t0) * 1e3)
    sc, sd = results["search"]
    same = (np.array_equal(np.array([c for c, _ in results["loop"]]), sc) and
            np.array_equal(np.array([d for _, d in results["loop"]]), sd))
    out["a"] = {"shape": {"frames": w.n_frames, "rays_per_frame": w.n_rays, "gyro_samples": int(ts.shape[0]),
                          "rotations": len(rots), "delays": int(D)},
                "results_bit_identical": bool(same),
                "ms_median": {k: float(np.median(v)) for k, v in t.items()},
                "ms_p10_p90": {k: [float(np.percentile(v, 10)), float(np.percentile(v, 90))] for k, v in t.items()},
                "reps": args.reps}
    med = out["a"]["ms_median"]
    out["a"]["speedup_vs_loop"] = med["loop"] / med["search"]
    out["a"]["grid_ms_per_rotation"] = (med["search"] - med["search_no_frames"]) / len(rots)
    p.close()
    loop.close()
    # ---- (b) ------------------------------------------------------------------------------------------
    libs = {"this": args.lib or pkg.LIB_PATH}
    if args.base_lib:
        libs["base"] = args.base_lib
    tmp = tempfile.mkdtemp(prefix="prof_rotation_search_")
    try:
        scene = os.path.join(tmp, "c2.npz")
        np.savez(scene, quats=w.quats, gyro_rate=w.gyro_rate, gyro_t0=w.gyro_t0, frame_ids=w.frame_ids,
                 ts_a=w.ts_a, ts_b=w.ts_b, rays_a=w.rays_a, rays_b=w.rays_b, ts=ts, omega=w.omega, step=step,
                 radius=radius)
        runs = {k: [] for k in libs}
        for rnd in range(args.rounds):
            order = list(libs.items())
            if rnd % 2:
                order.reverse()
            for k, lib in order:
                env = dict(os.environ, RSSYNC_B200_LIB=os.path.abspath(lib))
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--c5-child", scene, "--reps",
                                    str(args.reps)], env=env, capture_output=True, text=True, check=True)
                runs[k].append(json.loads(r.stdout.strip().splitlines()[-1]))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    c5 = {"variants": 48, "rounds": args.rounds, "reps_per_round": args.reps}
    for k, rs in runs.items():
        ms = [x for r in rs for x in r["ms"]]
        c5[k] = {"lib": rs[0]["lib"], "ms_median": float(np.median(ms)),
                 "ms_p10_p90": [float(np.percentile(ms, 10)), float(np.percentile(ms, 90))],
                 "round_medians": [float(np.median(r["ms"])) for r in rs]}
    if "base" in runs:
        c5["this_over_base"] = c5["this"]["ms_median"] / c5["base"]["ms_median"]
        c5["results_bit_identical"] = all(r["cost"] == runs["base"][0]["cost"] and r["delay"] == runs["base"][0]["delay"]
                                          for r in runs["this"] + runs["base"])
    out["b_c5"] = c5
    out["gpu_after"] = gpu_info()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "prof_rotation_search.json"), "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
