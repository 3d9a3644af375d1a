"""Track input from host numpy buffers against the same input from CUDA tensors (set_track_batch, which
dispatches to rssync_set_track_batch / rssync_set_track_batch_device), on the C2 (3300 x 200) and C3
(10000 x 500) shapes:

  * ingest: wall time of the bulk call, each ending in a device synchronise (median);
  * C2 end to end: SetGyroQuaternions + tracks + the 201-offset DebugPreSync-style curve read back,
    median of --steps steps after warm-up, the two forms alternating, L2 flushed (512 MB memset)
    before every step, outside the timed region;
  * the check-and-stage kernel alone, from torch.profiler in a separate pass, with the bytes it moves
    (reads and writes 64 B per ray, 32 B of offsets and verdicts per frame) and GB/s against the
    7.7 TB/s HBM3e data-sheet figure;
  * the GPU's name and power limit, read in the same run.

The device form's curve is checked bit for bit against the host form's at every shape.  Needs a CUDA
GPU and fails without one.  Prints the results as JSON; with --out DIR also writes them to
DIR/prof_device_ingest.json.

    python tools/prof_device_ingest.py [--out DIR] [--steps 20] [--reps 10]
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


def gpu_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0),
            "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None}


def load(pkg, w, bufs, stream):
    p = pkg.SyncProblem(seed=100)
    p.set_stream(stream.cuda_stream)
    p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
    p.set_track_batch(w.frame_ids, np.full(w.n_frames, w.n_rays), *bufs)
    p.flush()
    return p


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for prof_device_ingest.json (default: print only)")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("prof_device_ingest: no CUDA device (this measurement has no CPU form)")
    pkg = importlib.import_module("rs-sync_b200")
    synth = importlib.import_module("rs-sync_b200.synth")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)
    flush_buf = torch.empty(512 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    out = {"gpu": gpu_info(), "shapes": {}}
    for name in ("C2", "C3"):
        w = synth.make_workload(name, procs=min(16, os.cpu_count() or 1))
        F, N = w.n_frames, w.n_rays
        counts = np.full(F, N)
        host_bufs = (w.ts_a, w.ts_b, w.rays_a, w.rays_b)
        dev_bufs = tuple(torch.as_tensor(x.reshape(-1)).to(dev) for x in host_bufs)
        ph, pd = load(pkg, w, host_bufs, stream), load(pkg, w, dev_bufs, stream)
        fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
        delays = np.linspace(-w.presync_radius, w.presync_radius, 201)
        ch = ph.presync_grid(fb, fe, delays, stream=pkg.STREAM_DEBUG, call_no=5)
        cd = pd.presync_grid(fb, fe, delays, stream=pkg.STREAM_DEBUG, call_no=5)
        res = {"frames": F, "rays_per_frame": N, "curves_bit_identical": bool(np.array_equal(ch, cd))}
        # ---- ingest alone --------------------------------------------------------------------------
        t = {"host": [], "device": []}
        for i in range(args.reps + 2):
            for form, p, bufs in (("host", ph, host_bufs), ("device", pd, dev_bufs)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                p.set_track_batch(w.frame_ids, counts, *bufs)
                torch.cuda.synchronize()
                if i >= 2:
                    t[form].append((time.perf_counter() - t0) * 1e3)
        res["ingest_ms_median"] = {k: float(np.median(v)) for k, v in t.items()}
        res["ingest_ms_min"] = {k: float(np.min(v)) for k, v in t.items()}
        # ---- end to end (C2) -----------------------------------------------------------------------
        if name == "C2":
            t = {"host": [], "device": []}
            same = True
            for i in range(args.steps + 3):
                for form, p, bufs in (("host", ph, host_bufs), ("device", pd, dev_bufs)):
                    flush_buf.zero_()
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    p.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
                    p.set_track_batch(w.frame_ids, counts, *bufs)
                    c = p.presync_grid(fb, fe, delays, stream=pkg.STREAM_DEBUG, call_no=100 + i)
                    dt = (time.perf_counter() - t0) * 1e3
                    if i >= 3:
                        t[form].append(dt)
                    if form == "host":
                        c_host = c
                    else:
                        same = same and bool(np.array_equal(c, c_host))
            res["e2e_ms_median"] = {k: float(np.median(v)) for k, v in t.items()}
            res["e2e_ms_p10_p90"] = {k: [float(np.percentile(v, 10)), float(np.percentile(v, 90))] for k, v in t.items()}
            res["e2e_steps"] = args.steps
            res["e2e_curves_bit_identical"] = same
        out["shapes"][name] = res
        # ---- the check-and-stage kernel from torch.profiler (a pass of its own) ----------------------
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                pd.set_track_batch(w.frame_ids, counts, *dev_bufs)
            torch.cuda.synchronize()
        ev = [e for e in prof.events() if "stage_tracks_kernel" in e.name]
        us = [e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total for e in ev]
        if us:
            k_us = float(np.median(us))
            nbytes = 2 * 64 * F * N + 32 * F
            res["stage_kernel"] = {"launches_seen": len(us), "median_us": k_us, "bytes": nbytes,
                                   "GB_per_s": nbytes / (k_us * 1e-6) / 1e9,
                                   "share_of_7.7TB_per_s": nbytes / (k_us * 1e-6) / (HBM_TBS * 1e12)}
        else:
            res["stage_kernel"] = "not measured: the profiler listed no stage_tracks_kernel event"
        ph.close()
        pd.close()
        del dev_bufs
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "prof_device_ingest.json"), "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
