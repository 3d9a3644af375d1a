"""Rays with row fractions (SyncProblem.set_track_row_fractions, rssync_set_track_row_fractions(_device)): the
bulk call and the readout search on them against what an own-lens caller does without them, and the ingest
paths they share kernels with on two builds of the library.

  (a) C2 shape (3300 frames x 200 rays): one bulk call of 660 000 rays, ending in a device synchronise, in
      four forms alternating: set_track_row_fractions from host arrays and from CUDA tensors, against
      set_track_batch from host arrays and from CUDA tensors with the same timestamps formed beforehand.
      The frame tables are compared byte for byte.
  (b) C2, 11 candidate readouts (0 .. 2 x the synthetic readout), PreSync's delay grid of C2 (step 2 ms,
      radius 0.2 s: D = 200 offsets):
        * search: one readout_search call on the row-fractions frames (it ends in a device synchronise);
        * loop: per readout, ts = frame_ts + readout * frac formed on the host, set_track_batch into one
          problem, PreSync -- what a caller with its own lens model writes without the search.
      Medians over --reps repetitions, the forms alternating; (cost, delay) pairs checked bit for bit at the
      same RNG call numbers.
  (c) Regression of the touched kernels: set_track_batch and set_track_pixels (host and device forms) and
      the C2 end-to-end step (SetGyroQuaternions + set_track_batch + a 201-offset loss grid, as bench.py's
      single-GPU end-to-end step) in subprocesses that load the library named by --lib and by --base-lib
      (e.g. a build of the parent commit into another directory) through RSSYNC_B200_LIB, alternating,
      --rounds rounds of --reps repetitions each.  The two builds' loss curves are compared bit for bit.
  (d) the GPU's name, power limit and max SM clock, read in the same run.

Needs a CUDA GPU and fails without one.  Prints the results as JSON; with --out DIR also writes them to
DIR/prof_row_fractions.json.

    python tools/prof_row_fractions.py [--out DIR] [--reps 10] [--base-lib PATH] [--lib PATH] [--rounds 3]
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


def stats(v):
    return {"median": float(np.median(v)), "p10_p90": [float(np.percentile(v, 10)), float(np.percentile(v, 90))]}


def timed(forms, reps, sync):
    """alternate the forms; the first round warms every shape up.  Returns (ms lists, last results)"""
    t = {k: [] for k in forms}
    results = {}
    for i in range(reps + 1):
        for k, fn in forms.items():
            sync()
            t0 = time.perf_counter()
            results[k] = fn()
            sync()
            if i >= 1:
                t[k].append((time.perf_counter() - t0) * 1e3)
    return t, results


def regression_child(path, reps):
    """the ingest forms and the end-to-end step on the saved C2 scene, through a minimal ctypes binding of
    the library RSSYNC_B200_LIB names (entry points every build has, so a build of an older commit loads too)"""
    import ctypes as C
    import torch
    lib_path = os.environ["RSSYNC_B200_LIB"]
    L = C.CDLL(lib_path)
    P, dp, ip, sp = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_size_t)
    L.rssync_create.argtypes = [C.POINTER(P)]
    L.rssync_destroy.argtypes = [P]
    L.rssync_set_gyro_fixed.argtypes = [P, dp, C.c_size_t, C.c_double, C.c_double]
    L.rssync_set_track_batch.argtypes = [P, C.c_size_t, ip, sp, dp, dp, dp, dp]
    L.rssync_set_track_batch_device.argtypes = [P, C.c_size_t, ip, sp, P, P, P, P, P]
    L.rssync_set_track_pixels.argtypes = [P, C.c_size_t, ip, sp, dp, dp, dp, dp, dp, C.c_double]
    L.rssync_set_track_pixels_device.argtypes = [P, C.c_size_t, ip, sp, dp, dp, P, P, dp, C.c_double, P]
    L.rssync_presync_grid.argtypes = [P, C.c_int64, C.c_int64, dp, C.c_int, C.c_int, C.c_uint64, C.c_uint64, dp,
                                      C.POINTER(C.c_uint)]
    d = {k: np.ascontiguousarray(v) for k, v in np.load(path).items()}
    ptr = lambda a: a.ctypes.data_as(dp)  # noqa: E731
    F, N = d["ts_a"].shape
    ids = d["frame_ids"].astype(np.int64)
    counts = np.full(F, N, dtype=np.uint64)
    idp, cnp = ids.ctypes.data_as(ip), counts.ctypes.data_as(sp)
    fta, ftb = ids / float(d["fps"]), (ids + 1) / float(d["fps"])
    lens = np.ascontiguousarray(d["lens"])
    rows = float(d["rows"])
    dev = {k: torch.from_numpy(d[k]).cuda() for k in ("ts_a", "ts_b", "rays_a", "rays_b", "px_a", "px_b")}
    dv = {k: C.c_void_p(v.data_ptr()) for k, v in dev.items()}
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    fb, fe = int(ids[0]), int(ids[-1]) + 1
    delays = np.ascontiguousarray(d["delays"])
    curve = np.empty(delays.shape[0])
    flags = C.c_uint()
    probs = {}
    for k in ("batch_host", "batch_device", "pixels_host", "pixels_device", "e2e"):
        h = P()
        assert L.rssync_create(C.byref(h)) == 0
        assert L.rssync_set_gyro_fixed(h, ptr(d["quats"]), d["quats"].shape[0], float(d["gyro_rate"]),
                                       float(d["gyro_t0"])) == 0
        probs[k] = h

    def ok(rc):
        assert rc == 0, rc

    def e2e():
        h = probs["e2e"]
        ok(L.rssync_set_gyro_fixed(h, ptr(d["quats"]), d["quats"].shape[0], float(d["gyro_rate"]),
                                   float(d["gyro_t0"])))
        ok(L.rssync_set_track_batch(h, F, idp, cnp, ptr(d["ts_a"]), ptr(d["ts_b"]), ptr(d["rays_a"]),
                                    ptr(d["rays_b"])))
        ok(L.rssync_presync_grid(h, fb, fe, ptr(delays), delays.shape[0], 2, 7, 0, ptr(curve), C.byref(flags)))

    forms = {
        "set_track_batch_host": lambda: ok(L.rssync_set_track_batch(
            probs["batch_host"], F, idp, cnp, ptr(d["ts_a"]), ptr(d["ts_b"]), ptr(d["rays_a"]), ptr(d["rays_b"]))),
        "set_track_batch_device": lambda: ok(L.rssync_set_track_batch_device(
            probs["batch_device"], F, idp, cnp, dv["ts_a"], dv["ts_b"], dv["rays_a"], dv["rays_b"], stream)),
        "set_track_pixels_host": lambda: ok(L.rssync_set_track_pixels(
            probs["pixels_host"], F, idp, cnp, ptr(fta), ptr(ftb), ptr(d["px_a"]), ptr(d["px_b"]), ptr(lens), rows)),
        "set_track_pixels_device": lambda: ok(L.rssync_set_track_pixels_device(
            probs["pixels_device"], F, idp, cnp, ptr(fta), ptr(ftb), dv["px_a"], dv["px_b"], ptr(lens), rows, stream)),
        "c2_e2e_step": e2e,
    }
    t, _ = timed(forms, reps, torch.cuda.synchronize)
    for h in probs.values():
        L.rssync_destroy(h)
    print(json.dumps({"lib": os.path.relpath(lib_path, ROOT), "ms": t, "curve": curve.tolist()}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for prof_row_fractions.json (default: print only)")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3, help="(c): alternating rounds per library")
    ap.add_argument("--lib", default=None, help="(c): this build (default: the package's library)")
    ap.add_argument("--base-lib", default=None, help="(c): the build to compare against (default: none)")
    ap.add_argument("--child", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:
        return regression_child(args.child, args.reps)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("prof_row_fractions: no CUDA device (this measurement has no CPU form)")
    pkg = importlib.import_module("rs-sync_b200")
    synth = importlib.import_module("rs-sync_b200.synth")
    out = {"gpu": gpu_info()}
    w = synth.make_workload("C2", procs=min(16, os.cpu_count() or 1))
    F, N = w.n_frames, w.n_rays
    ids = w.frame_ids
    counts = np.full(F, N, dtype=np.uint64)
    fb, fe = int(ids[0]), int(ids[-1]) + 1
    fta, ftb = ids / w.fps, (ids + 1) / w.fps
    qa, qb = np.ascontiguousarray(w.px_a[..., 1] / synth.HEIGHT), np.ascontiguousarray(w.px_b[..., 1] / synth.HEIGHT)
    R = synth.READOUT
    tsa = np.repeat(fta, N).reshape(F, N) + R * qa
    tsb = np.repeat(ftb, N).reshape(F, N) + R * qb
    assert np.array_equal(tsa, w.ts_a) and np.array_equal(tsb, w.ts_b)
    cuda = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in
            (("qa", qa), ("qb", qb), ("ts_a", w.ts_a), ("ts_b", w.ts_b), ("rays_a", w.rays_a), ("rays_b", w.rays_b))}
    initial, step, radius = 0.0, w.presync_step, w.presync_radius
    D = pkg.presync_delays(initial, step, radius).shape[0]

    def problem():
        p = pkg.SyncProblem(seed=100)
        p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
        return p

    # ---- (a) ------------------------------------------------------------------------------------------
    pa = {k: problem() for k in ("rows_host", "rows_device", "batch_host", "batch_device")}
    c = cuda
    forms = {
        "set_track_row_fractions_host": lambda: pa["rows_host"].set_track_row_fractions(
            ids, counts, fta, ftb, qa, qb, w.rays_a, w.rays_b, R),
        "set_track_row_fractions_device": lambda: pa["rows_device"].set_track_row_fractions(
            ids, counts, fta, ftb, c["qa"], c["qb"], c["rays_a"], c["rays_b"], R),
        "set_track_batch_host": lambda: pa["batch_host"].set_track_batch(
            ids, counts, w.ts_a, w.ts_b, w.rays_a, w.rays_b),
        "set_track_batch_device": lambda: pa["batch_device"].set_track_batch(
            ids, counts, c["ts_a"], c["ts_b"], c["rays_a"], c["rays_b"]),
    }
    t, _ = timed(forms, args.reps, torch.cuda.synchronize)
    tables = {k: p.frame_table().tobytes() for k, p in pa.items()}
    out["a_bulk_call"] = {"shape": {"frames": F, "rays_per_frame": N, "rays": F * N},
                          "frame_tables_identical": len(set(tables.values())) == 1,
                          "ms": {k: stats(v) for k, v in t.items()}, "reps": args.reps}
    for p in pa.values():
        p.close()
    # ---- (b) ------------------------------------------------------------------------------------------
    readouts = np.linspace(0.0, 2.0 * R, 11)
    calls = np.arange(len(readouts), dtype=np.uint64) + 50
    src = problem()
    src.set_track_row_fractions(ids, counts, fta, ftb, qa, qb, w.rays_a, w.rays_b, R)
    src.flush()
    loop = problem()

    def run_search():
        return src.readout_search(readouts, initial, fb, fe, step, radius, call_nos=calls)

    def run_loop():
        res = []
        for r, cn in zip(readouts, calls):
            ta = np.repeat(fta, N).reshape(F, N) + r * qa
            tb = np.repeat(ftb, N).reshape(F, N) + r * qb
            loop.set_track_batch(ids, counts, ta, tb, w.rays_a, w.rays_b)
            loop.set_rng(100, int(cn))
            res.append(loop.PreSync(initial, fb, fe, step, radius))
        return res

    t, results = timed({"search": run_search, "loop": run_loop}, args.reps, torch.cuda.synchronize)
    sc, sd = results["search"]
    same = (np.array_equal(np.array([x for x, _ in results["loop"]]), sc) and
            np.array_equal(np.array([y for _, y in results["loop"]]), sd))
    out["b_readout_search"] = {"shape": {"frames": F, "rays_per_frame": N, "readouts": len(readouts), "delays": int(D)},
                               "results_bit_identical": bool(same),
                               "ms": {k: stats(v) for k, v in t.items()}, "reps": args.reps}
    med = {k: float(np.median(v)) for k, v in t.items()}
    out["b_readout_search"]["speedup_vs_loop"] = med["loop"] / med["search"]
    src.close()
    loop.close()
    # ---- (c) ------------------------------------------------------------------------------------------
    libs = {"this": args.lib or pkg.LIB_PATH}
    if args.base_lib:
        libs["base"] = args.base_lib
    tmp = tempfile.mkdtemp(prefix="prof_row_fractions_")
    try:
        scene = os.path.join(tmp, "c2.npz")
        np.savez(scene, quats=w.quats, gyro_rate=w.gyro_rate, gyro_t0=w.gyro_t0, frame_ids=w.frame_ids, fps=w.fps,
                 ts_a=w.ts_a, ts_b=w.ts_b, rays_a=w.rays_a, rays_b=w.rays_b, px_a=w.px_a, px_b=w.px_b,
                 lens=np.array(synth.LENS, dtype=np.float64), rows=float(synth.HEIGHT),
                 delays=np.linspace(-w.presync_radius, w.presync_radius, 201))
        runs = {k: [] for k in libs}
        for rnd in range(args.rounds):
            order = list(libs.items())
            if rnd % 2:
                order.reverse()
            for k, lib in order:
                env = dict(os.environ, RSSYNC_B200_LIB=os.path.abspath(lib))
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", scene, "--reps",
                                    str(args.reps)], env=env, capture_output=True, text=True, check=True)
                runs[k].append(json.loads(r.stdout.strip().splitlines()[-1]))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    reg = {"rounds": args.rounds, "reps_per_round": args.reps}
    for k, rs in runs.items():
        reg[k] = {"lib": rs[0]["lib"]}
        for form in rs[0]["ms"]:
            ms = [x for r in rs for x in r["ms"][form]]
            reg[k][form] = dict(stats(ms), round_medians=[float(np.median(r["ms"][form])) for r in rs])
    if "base" in runs:
        reg["this_over_base"] = {f: reg["this"][f]["median"] / reg["base"][f]["median"] for f in runs["this"][0]["ms"]}
        reg["e2e_curves_bit_identical"] = all(r["curve"] == runs["base"][0]["curve"] for r in runs["this"] + runs["base"])
    out["c_regression"] = reg
    out["gpu_after"] = gpu_info()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "prof_row_fractions.json"), "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
