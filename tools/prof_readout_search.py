"""Rolling-shutter readout search (SyncProblem.readout_search, rssync_readout_search) against the loop a
caller writes without it, on the C2 shape (3300 frames x 200 pixel pairs), 11 candidate readouts and
PreSync's delay grid of C2 (step 2 ms, radius 0.2 s: D = 200 offsets):

  * search: one readout_search call over the 11 readouts (it ends in a device synchronise);
  * loop, fresh: per readout a new problem, SetGyroQuaternions, set_track_pixels from host arrays with
    the readout in the lens, PreSync -- what a caller does today;
  * loop, reuse: per readout set_track_pixels from host arrays into one problem (frames replaced in
    place) and PreSync;
  * retime_frames_kernel alone, from torch.profiler in a pass of its own, with the bytes it moves and
    its share of one search step (re-time + grid);
  * the GPU's name, power limit and max SM clock, read in the same run.

Medians over --reps repetitions, the three forms alternating.  The arena (42 MB) fits the L2; it is not
flushed between calls.  The search's (cost, delay) pairs are checked bit for bit against the loop's at
the same RNG call numbers.  Needs a CUDA GPU and fails without one.  Prints the results as JSON; with
--out DIR also writes them to DIR/prof_readout_search.json.

With --devices 0,1,2,3 it times instead the same search on one problem spread over those devices
(rssync_create_multi, readouts sharded by device) against the problem on the first device alone:

  * one_device: readout_search on the single-device problem;
  * multi_repeat: readout_search on the multi-device problem whose replicas already hold the row fractions;
  * multi_first: the same right after a re-ingest of the same pixels (in place), once a PreSync grid has
    sent the arena on: the search sends the row-fraction plane first (one grouped broadcast).

The three alternate; medians over --reps.  Results (curves included) are checked bit for bit against the
single-device search, the bytes and collectives of the plane's broadcast are read from the problem's
statistics, and the card's name, power limit and max SM clock are read for every device used.  Written to
DIR/prof_readout_search_<G>gpu.json with --out.

    python tools/prof_readout_search.py [--out DIR] [--reps 10] [--devices 0,1,2,3]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_TBS = 7.7  # HGX B200 data sheet, one GPU


def gpu_info(device=0):
    import torch
    q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(device),
            "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None}


def multi_main(args, pkg, synth, w, devices):
    """the readout search on a multi-device problem against the same problem on devices[0]"""
    import torch
    F, N = w.n_frames, w.n_rays
    counts = np.full(F, N)
    ta, tb = w.frame_ids / w.fps, (w.frame_ids + 1) / w.fps
    pa, pb = w.px_a.reshape(-1), w.px_b.reshape(-1)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    initial, step, radius = 0.0, w.presync_step, w.presync_radius
    delays = pkg.presync_delays(initial, step, radius)
    readouts = np.linspace(0.0, 0.02, 11)
    calls = np.arange(len(readouts), dtype=np.uint64) + 50
    lens = (float(synth.READOUT),) + tuple(synth.LENS[1:])

    def make(devs):
        p = pkg.SyncProblem(seed=100, devices=devs)
        p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
        p.set_track_pixels(w.frame_ids, counts, ta, tb, pa, pb, lens, synth.HEIGHT)
        return p

    one, many = make([devices[0]]), make(devices)
    assert many.device_count() == len(devices)
    many.presync_grid(fb, fe, delays[:8], call_no=1)  # the arena goes out here, not inside the timed search

    def sync_all():
        for d in devices:
            torch.cuda.synchronize(d)

    def search(p):
        return p.readout_search(readouts, initial, fb, fe, step, radius, call_nos=calls, curves=True)

    def first():
        many.set_track_pixels(w.frame_ids, counts, ta, tb, pa, pb, lens, synth.HEIGHT)  # in place: the plane is stale
        many.presync_grid(fb, fe, delays[:8], call_no=1)
        sync_all()
        s0 = many.stats()
        t0 = time.perf_counter()
        out = search(many)
        sync_all()
        ms = (time.perf_counter() - t0) * 1e3
        s1 = many.stats()
        return out, ms, (s1["broadcast_bytes"] - s0["broadcast_bytes"], s1["nccl_calls"] - s0["nccl_calls"])

    def timed(p):
        sync_all()
        t0 = time.perf_counter()
        out = search(p)
        sync_all()
        return out, (time.perf_counter() - t0) * 1e3

    t = {"one_device": [], "multi_repeat": [], "multi_first": []}
    want, same, plane = None, True, None
    for i in range(args.reps + 1):
        want, ms1 = timed(one)
        got_first, msf, plane = first()
        got, msr = timed(many)
        same = same and all(np.array_equal(a, b) for a, b in zip(want, got)) and \
            all(np.array_equal(a, b) for a, b in zip(want, got_first))
        if i >= 1:  # the first round warms every shape up
            t["one_device"].append(ms1)
            t["multi_first"].append(msf)
            t["multi_repeat"].append(msr)
    arena = many.device_state()["arena_rays"]
    G = len(devices)
    out = {"gpus": [gpu_info(d) for d in devices], "devices": list(devices),
           "shape": {"frames": F, "pixel_pairs_per_frame": N, "readouts": len(readouts), "delays": int(delays.size),
                     "arena_rays": int(arena)},
           "results_bit_identical": bool(same),
           "plane_broadcast": {"bytes": int(plane[0]), "collectives": int(plane[1]),
                               "expected_bytes": 16 * int(arena) if G > 1 else 0},
           "rounds": -(-len(readouts) // G),
           "ms_median": {k: float(np.median(v)) for k, v in t.items()},
           "ms_p10_p90": {k: [float(np.percentile(v, 10)), float(np.percentile(v, 90))] for k, v in t.items()},
           "reps": args.reps}
    out["speedup_repeat_vs_one_device"] = out["ms_median"]["one_device"] / out["ms_median"]["multi_repeat"]
    out["plane_cost_ms"] = out["ms_median"]["multi_first"] - out["ms_median"]["multi_repeat"]
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, f"prof_readout_search_{G}gpu.json"), "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for prof_readout_search.json (default: print only)")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--devices", default=None,
                    help="comma-separated CUDA devices: time the search on one problem spread over them")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("prof_readout_search: no CUDA device (this measurement has no CPU form)")
    pkg = importlib.import_module("rs-sync_b200")
    synth = importlib.import_module("rs-sync_b200.synth")
    w = synth.make_workload("C2", procs=min(16, os.cpu_count() or 1))
    if args.devices:
        devices = [int(d) for d in args.devices.split(",")]
        if len(devices) > torch.cuda.device_count():
            raise SystemExit(f"prof_readout_search: {len(devices)} devices asked, {torch.cuda.device_count()} present")
        return multi_main(args, pkg, synth, w, devices)
    F, N = w.n_frames, w.n_rays
    counts = np.full(F, N)
    ta, tb = w.frame_ids / w.fps, (w.frame_ids + 1) / w.fps
    pa, pb = w.px_a.reshape(-1), w.px_b.reshape(-1)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    initial, step, radius = 0.0, w.presync_step, w.presync_radius
    D = pkg.presync_delays(initial, step, radius).shape[0]
    readouts = np.linspace(0.0, 0.02, 11)
    calls = np.arange(len(readouts), dtype=np.uint64) + 50

    def lens(r):
        return (float(r),) + tuple(synth.LENS[1:])

    def fresh(r):
        p = pkg.SyncProblem(seed=100)
        p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
        p.set_track_pixels(w.frame_ids, counts, ta, tb, pa, pb, lens(r), synth.HEIGHT)
        return p

    src = fresh(synth.READOUT)
    reuse = fresh(synth.READOUT)

    def run_search():
        return src.readout_search(readouts, initial, fb, fe, step, radius, call_nos=calls)

    def run_fresh():
        out = []
        for r, c in zip(readouts, calls):
            p = fresh(r)
            p.set_rng(100, int(c))
            out.append(p.PreSync(initial, fb, fe, step, radius))
            p.close()
        return out

    def run_reuse():
        out = []
        for r, c in zip(readouts, calls):
            reuse.set_track_pixels(w.frame_ids, counts, ta, tb, pa, pb, lens(r), synth.HEIGHT)
            reuse.set_rng(100, int(c))
            out.append(reuse.PreSync(initial, fb, fe, step, radius))
        return out

    forms = {"search": run_search, "loop_fresh": run_fresh, "loop_reuse": run_reuse}
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
    same = all(np.array_equal(np.array([c for c, _ in results[k]]), sc) and
               np.array_equal(np.array([d for _, d in results[k]]), sd) for k in ("loop_fresh", "loop_reuse"))
    out = {"gpu": gpu_info(), "shape": {"frames": F, "pixel_pairs_per_frame": N, "readouts": len(readouts),
                                        "delays": int(D)},
           "results_bit_identical": bool(same),
           "ms_median": {k: float(np.median(v)) for k, v in t.items()},
           "ms_p10_p90": {k: [float(np.percentile(v, 10)), float(np.percentile(v, 90))] for k, v in t.items()},
           "reps": args.reps}
    out["speedup_vs_loop_fresh"] = out["ms_median"]["loop_fresh"] / out["ms_median"]["search"]
    out["speedup_vs_loop_reuse"] = out["ms_median"]["loop_reuse"] / out["ms_median"]["search"]
    # ---- retime_frames_kernel and the grid from torch.profiler (a pass of its own) ---------------------
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            run_search()
        torch.cuda.synchronize()

    def device_us(e):
        return e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total

    rt = [device_us(e) for e in prof.events() if "retime_frames_kernel" in e.name]
    grid = [device_us(e) for e in prof.events() if "presync_kernel" in e.name]
    if rt:
        k_us = float(np.median(rt))
        pad = (N + 31) // 32 * 32
        # reads: 6 ray fields (48 B) + orig (4 B) + row fractions (16 B) per ray, a 32 B record per frame;
        # writes: the padded tiles (64 B) + orig / pos (8 B) per ray slot
        nbytes = F * N * 68 + F * 32 + F * pad * 72
        out["retime_kernel"] = {"launches_seen": len(rt), "median_us": k_us, "bytes": nbytes,
                                "GB_per_s": nbytes / (k_us * 1e-6) / 1e9,
                                "share_of_7.7TB_per_s": nbytes / (k_us * 1e-6) / (HBM_TBS * 1e12)}
        if grid:
            g_us = float(np.median(grid))
            out["grid_kernel_median_us"] = g_us
            out["retime_share_of_step"] = k_us / (k_us + g_us)
    else:
        out["retime_kernel"] = "not measured: the profiler listed no retime_frames_kernel event"
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "prof_readout_search.json"), "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
