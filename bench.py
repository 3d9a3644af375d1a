#!/usr/bin/env python
"""Benchmark of the rs-sync loss engine on B200 (contract: see DESIGN.md §7).

A "step" is one pass of the PreSync brute-force grid (offset x frame x feature loss
evaluations, the body of pre_sync, core_private.cpp:61-90 of the reference) over the
GX012440-shaped synthetic workload C2 of BASELINE.json: frames 3900..7199 (3300) x 200 rays x
201 offsets (DebugPreSync's linspace grid, radius 200 ms).  With N > 1 GPUs every rank holds a
replica of the inputs and evaluates its own 201-offset slice of a grid N times as wide
(weak scaling, radius 0.2*N s, same 2 ms step); only the loss-curve slices are gathered (NCCL).

    python bench.py --gpus N --steps K --warmup W            # the B200 engine
    python bench.py --impl reference --steps K --warmup W    # the CPU path on the host cores
    python bench.py --steps K --warmup W --dump-outputs DIR  # also save the last timed step's curve

The inputs are generated from fixed seeds and every grid call's RNG is keyed by its call number, so
two runs with the same arguments compute on identical inputs and their dumps can be compared.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FLOP_PER_CELL = 285.0     # SURVEY.md §8(d): algorithmic FP64 flop per (offset, frame, ray) cell
OFFSETS_PER_GPU = 201
METRIC = "presync_loss_evals_per_s"
UNIT = "cells/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the headline grid and of the end-to-end path (the syncpoint and scale "
                         "sections report the best of a fixed number of whole passes)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C2")
    ap.add_argument("--no-sync", action="store_true", help="skip the syncpoints/s section")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline section")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--scale-configs", action="store_true", help="(kept for old command lines: now the default)")
    ap.add_argument("--no-scale", action="store_true",
                    help="skip C3 (strong scaling) and C4 with 900 syncpoints (about 25 s at N = 1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the loss curve of the last one (float64, one value per "
                         "offset of the whole grid) to DIR/presync_costs.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return a


def make_workload(name, n_gpus):
    synth = importlib.import_module("rs-sync_b200.synth")
    # weak scaling widens the grid with the GPU count (radius 0.2 s per GPU); the gyro track is
    # generated for the widest case (8 GPUs) at every N, so the scene -- and with it the syncpoint
    # loop's results -- are the same for every N
    radius = 0.2 * n_gpus if name in ("C1", "C2") else None
    w = synth.make_workload(name, radius=radius, gyro_pad_radius=1.6 if name in ("C1", "C2") else None)
    return w


def grid_delays(w, n_gpus):
    n = OFFSETS_PER_GPU * n_gpus
    r = w.presync_radius
    return np.array([0.0 - r + 2 * r * i / (n - 1) for i in range(n)])  # core_private.cpp:345


def workload_name(w, n_gpus):
    return (f"{w.name}: synthetic GoPro-shaped, frames {int(w.frame_ids[0])}..{int(w.frame_ids[-1])} "
            f"({w.n_frames}) x {w.n_rays} rays x {OFFSETS_PER_GPU * n_gpus} offsets "
            f"(DebugPreSync linspace, radius {w.presync_radius * 1e3:.0f} ms, {OFFSETS_PER_GPU} offsets per GPU)")


# ------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 8:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for nm, val in zip(names, p[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        top = sorted(sm)[len(sm) // 2:]  # samples under load are the upper half
        return {"sm_mhz": float(np.median(top)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------
def cpu_problem(w, threads, prefer_ref=True):
    """The CPU arm: the unmodified reference compiled against the shim when oracle/_ref exists,
    else the oracle port.  Returns (problem, kind)."""
    from oracle import loader
    if prefer_ref:
        try:
            from oracle import ref_loader
            if ref_loader.available():
                p = ref_loader.RefProblem(threads=threads, seed=100)
                p.load(w)
                return p, "reference"
        except Exception:
            pass
    p = loader.OracleProblem(threads=threads, seed=100).load(w)
    return p, "port"


def cpu_sample_shape(w, delays, cells_per_s, seconds):
    """frames x offsets sample of the workload that takes about `seconds` on the CPU arm."""
    want = max(cells_per_s * seconds, 1.0)
    n_off = int(max(1, min(len(delays), want // (w.n_frames * w.n_rays))))
    return n_off


def time_cpu(p, w, delays, n_off, call_no=0):
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    lo = (len(delays) - n_off) // 2  # a contiguous, centred block of the grid (still a linspace)
    t = time.perf_counter()
    p.presync_grid(fb, fe, delays[lo:lo + n_off], stream=2, call_no=call_no)
    dt = time.perf_counter() - t
    return n_off * w.n_frames * w.n_rays / dt, dt


def cpu_baseline(w, delays, seconds):
    threads = os.cpu_count() or 1
    p, kind = cpu_problem(w, threads)
    rate, _ = time_cpu(p, w, delays, 1)                     # calibration (also warms the caches)
    n_off = cpu_sample_shape(w, delays, rate, seconds)
    rate, dt = time_cpu(p, w, delays, n_off)
    return {"value": rate, "unit": UNIT, "cores": threads, "kind": kind,
            "sample": f"{n_off} of {len(delays)} offsets x all {w.n_frames} frames x {w.n_rays} rays "
                      f"({n_off * w.n_frames * w.n_rays:.3g} cells, {dt:.1f} s)"}


def full_size_parity(prob, w, delays, pkg):
    """The checker at the bench's full frame count: a few offsets of the timed grid recomputed by the
    oracle port (same arithmetic contract and RNG keys) and compared with the engine's values."""
    from oracle import loader
    threads = os.cpu_count() or 1
    o = loader.OracleProblem(threads=threads, seed=100).load(w)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    pick = [0, len(delays) // 2, len(delays) - 1]
    worst = 0.0
    for i in pick:
        g = prob.presync_grid(fb, fe, delays[i:i + 1], stream=pkg.STREAM_DEBUG, call_no=77, offset_index_base=i)
        c = o.presync_grid(fb, fe, delays[i:i + 1], stream=2, call_no=77, offset_index_base=i)
        worst = max(worst, abs(float(g[0]) - float(c[0])) / abs(float(c[0])))
    return {"offsets_checked": len(pick), "frames": w.n_frames, "max_rel_err_vs_oracle": worst, "tolerance": 1e-9,
            "ok": bool(worst <= 1e-9)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = make_workload(args.workload, args.gpus)
    delays = grid_delays(w, args.gpus)
    threads = os.cpu_count() or 1
    p, kind = cpu_problem(w, threads)
    rate, _ = time_cpu(p, w, delays, 1)
    budget = min(20.0, 100.0 / max(1, args.steps + args.warmup))  # seconds of CPU work per step
    budget = float(os.environ.get("RSSYNC_REF_BUDGET", budget))   # (the CPU test suite shortens it)
    n_off = cpu_sample_shape(w, delays, rate, budget)
    for i in range(args.warmup):
        time_cpu(p, w, delays, n_off, call_no=i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        time_cpu(p, w, delays, n_off, call_no=100 + i)
    dt = time.perf_counter() - t0
    cells = n_off * w.n_frames * w.n_rays * args.steps
    value = cells / dt
    sample = (f"{n_off} of {len(delays)} offsets x all {w.n_frames} frames x {w.n_rays} rays per step")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(w, args.gpus), "step": "bounded sample: " + sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------
E_ROW, E_LOSS, E_GRAD = 145.0, 10.0, 14.0   # SURVEY 8(d): flop per (frame, ray) row build / loss cell / gradient
E_EST = lambda iters: 8.0 + 6.0 * iters + 2.0  # row normalisation + iters x (dot3, square) + hypothesis set-up


def host_wait(rank, key):
    """rank 0 has finished a solo measurement: release the other ranks, which wait on the host (the
    c10d store) rather than inside an NCCL barrier's spinning kernel"""
    import torch.distributed as dist
    store = dist.distributed_c10d._get_default_store()
    if rank == 0:
        store.set("rssync_" + key, "1")
    else:
        store.wait(["rssync_" + key])


def sync_flops(acc, n_rays, presync_cells):
    """algorithmic FP64 flop of a syncpoint loop from the engine's evaluation counters"""
    return (FLOP_PER_CELL * presync_cells +
            n_rays * (E_ROW * acc["sync_row_builds"] + E_LOSS * acc["sync_loss_evals"] +
                      (E_LOSS + E_GRAD) * acc["sync_lbfgs_evals"] + E_EST(200) * acc["sync_init_tasks"]))


def syncpoint_loop(prob, sps, win, step, radius, idx, n_total):
    """core_testcode.cpp:303-316 for the syncpoints idx (indices into sps): PreSync on every window in
    one grid launch, then 4 chained Sync calls advanced as batches.  Call numbers are those of ONE
    problem running all n_total syncpoints (PreSync s -> s, Sync round r -> n_total (r + 1) + s), so any
    sharding of idx over ranks computes the same numbers.  Returns (delays, costs, counters)."""
    idx = np.asarray(idx, dtype=np.int64)
    acc = {k: 0 for k in ("sync_row_builds", "sync_loss_evals", "sync_lbfgs_evals", "sync_init_tasks", "sync_outer_total")}
    if idx.size == 0:
        return np.empty(0), np.empty(0), acc
    fbs = np.asarray(sps, dtype=np.int64)[idx]
    _, d = prob.presync_windows(0.0, fbs, fbs + win, step, radius, call_nos=idx.astype(np.uint64))
    c = None
    for r in range(4):
        c, d = prob.sync_batch(d, fbs, fbs + win, 0.0, radius, call_nos=(n_total * (r + 1) + idx).astype(np.uint64))
        st = prob.stats()
        for k in acc:
            acc[k] += int(st[k])
    return d, c, acc


def bench_syncpoints(prob, w, label, rank, world, barrier, dev, fp64_peak, repeat=1):
    """syncpoints/s of the whole syncpoint loop of workload w, syncpoints sharded round-robin over the
    ranks, with the evaluation accounting of SURVEY 8(d) and, for N > 1, a comparison of the gathered
    result with rank 0 computing everything alone."""
    import torch
    import torch.distributed as dist
    sharded = importlib.import_module("rs-sync_b200.sharded")
    sps = w.syncpoints()
    S, win = len(sps), w.sync_window
    mine = np.arange(rank, S, world)
    syncpoint_loop(prob, sps, win, w.presync_step, 0.2, mine, S)  # warm-up (streams, graphs, first use)
    best = None
    for _ in range(repeat):
        barrier()
        t0 = time.perf_counter()
        d, c, acc = syncpoint_loop(prob, sps, win, w.presync_step, 0.2, mine, S)
        if world > 1:  # the one exchange: (cost, delay) of every syncpoint to every rank
            both = sharded._gather_rows(np.stack([c, d], axis=1), [len(range(r, S, world)) for r in range(world)],
                                        world, dev, dist)
            order = np.concatenate([np.arange(r, S, world) for r in range(world)])
            allc, alld = np.empty(S), np.empty(S)
            allc[order], alld[order] = both[:, 0], both[:, 1]
        else:
            allc, alld = c, d
        barrier()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    t = torch.tensor([best], dtype=torch.float64, device=dev)
    cnt = torch.tensor([float(acc[k]) for k in sorted(acc)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    acc = {k: int(v) for k, v in zip(sorted(acc), cnt.cpu().tolist())}
    secs = float(t[0])
    presync_cells = S * win * w.n_rays * len(importlib.import_module("rs-sync_b200").presync_delays(0.0, w.presync_step, 0.2))
    flops = sync_flops(acc, w.n_rays, presync_cells)
    true = np.array([w.true_delay_at(p) for p in sps])
    out = {"metric": "sync_syncpoints_per_s", "config": label, "value": S / secs, "unit": "syncpoints/s",
           "syncpoints": S, "seconds": secs,
           "what": "per syncpoint: PreSync(radius 200 ms, step 2 ms) on a 60-frame window + 4 chained Sync; "
                   "Sync calls batched across syncpoints, syncpoints sharded round-robin over the GPUs",
           "mean_abs_delay_error_ms": float(np.mean(np.abs(alld - true)) * 1e3),
           "row_builds": acc["sync_row_builds"], "loss_evals": acc["sync_loss_evals"],
           "lbfgs_evals": acc["sync_lbfgs_evals"], "init_estimates": acc["sync_init_tasks"],
           "outer_iters": acc["sync_outer_total"], "presync_cells": presync_cells,
           "algorithmic_gflop": flops / 1e9, "tflops": flops / secs / 1e12,
           "frac_fp64_peak": flops / secs / 1e12 / (fp64_peak * world) if fp64_peak > 0 else None,
           "checksum": float(np.sum(alld) + np.sum(allc) * 1e-6)}
    if world > 1:  # every N must compute the single-GPU numbers: rank 0 recomputes all of them alone
        ok = True
        n1 = None
        if rank == 0:
            for _ in range(repeat):  # the same best-of as the sharded run
                t1 = time.perf_counter()
                d1, c1, _ = syncpoint_loop(prob, sps, win, w.presync_step, 0.2, np.arange(S), S)
                dt1 = time.perf_counter() - t1
                n1 = dt1 if n1 is None else min(n1, dt1)
            ok = bool(np.array_equal(d1, alld) and np.array_equal(c1, allc))
        host_wait(rank, "sync_solo_" + label[:2])
        barrier()
        out["equals_one_gpu"] = ok
        out["n1_seconds_same_run"] = n1
        out["speedup_vs_one_gpu_same_run"] = (n1 / secs) if n1 else None
    return out, alld


def sync_parity_vs_oracle(w, alld, n_check=2):
    """the oracle port's sequential PreSync + 4 x Sync on the first syncpoints, same call numbers, against
    the engine's delays; also the CPU arm of syncpoints/s"""
    from oracle import loader
    threads = os.cpu_count() or 1
    sps = w.syncpoints()
    S, win = len(sps), w.sync_window
    worst, secs = 0.0, []
    for s in range(min(n_check, S)):
        pos = sps[s]
        o = loader.OracleProblem(threads=threads, seed=100).load_range(w, pos, win + 1)
        t = time.perf_counter()
        o.set_rng(100, s)
        d = o.PreSync(0.0, pos, pos + win, w.presync_step, 0.2)[1]
        for r in range(4):
            o.set_rng(100, S * (r + 1) + s)
            d = o.Sync(d, pos, pos + win, 0.0, 0.2)[1]
        secs.append(time.perf_counter() - t)
        worst = max(worst, abs(d - float(alld[s])) / abs(d))
    return ({"syncpoints_checked": min(n_check, S), "max_rel_err_vs_oracle": worst, "tolerance": 1e-9, "ok": bool(worst <= 1e-9)},
            {"value": 1.0 / float(np.mean(secs)), "unit": "syncpoints/s", "cores": threads, "kind": "port",
             "sample": f"{len(secs)} of {S} syncpoints ({float(np.mean(secs)):.2f} s each)"})


def read_traffic():
    """DRAM bytes of one launch of the dominant kernel, from the tracked ncu capture"""
    try:
        with open(os.path.join(ROOT, "profiles", "presync_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


def run_b200(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = max(args.gpus, world)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    cores = max(1, (os.cpu_count() or 1))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        # one process per GPU on one host, and the inputs enter through rank 0 only: its ingest thread
        # pool gets the cores the other ranks' (waiting) main threads leave, theirs get two
        share = max(2, cores - (local_world - 1)) if rank == 0 else 2
        os.environ.setdefault("RSSYNC_HOST_THREADS", str(share))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    pkg = importlib.import_module("rs-sync_b200")
    sharded = importlib.import_module("rs-sync_b200.sharded")
    w = make_workload(args.workload, n_gpus)
    delays = grid_delays(w, n_gpus)
    lo, hi = OFFSETS_PER_GPU * rank, OFFSETS_PER_GPU * (rank + 1)
    if world == 1:
        lo, hi = 0, len(delays)
    fb, fe = int(w.frame_ids[0]), int(w.frame_ids[-1]) + 1
    cells_per_step_rank = (hi - lo) * w.n_frames * w.n_rays
    cells_per_step = len(delays) * w.n_frames * w.n_rays

    stream = torch.cuda.current_stream()
    prob = pkg.SyncProblem(seed=100)
    prob.set_stream(stream.cuda_stream)
    prob.set_kernel_timing(True)
    prob.load(w, bulk=True)
    prob.flush()

    flush_buf = torch.empty(512 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # 512 MB > 126 MB L2
    gather_in = torch.empty(hi - lo, dtype=torch.float64, device=dev)
    gather_out = torch.empty((world, hi - lo), dtype=torch.float64, device=dev)

    def step(call_no, marks=None):
        costs = prob.presync_grid(fb, fe, delays[lo:hi], stream=pkg.STREAM_DEBUG, call_no=call_no,
                                  offset_index_base=lo)
        if marks is not None:
            marks.append(time.perf_counter())
        if world > 1:  # the only exchange: loss-curve slices
            gather_in.copy_(torch.from_numpy(costs))
            dist.all_gather_into_tensor(gather_out, gather_in)
            curve = gather_out.reshape(-1)
        else:
            curve = torch.from_numpy(costs)
        step.curve = curve.clone()
        return int(torch.argmin(curve))

    sampler = ClockSampler(local)
    sampler.start()  # nvidia-smi takes a moment to start: begin before the warm-up, keep the loaded half
    for i in range(args.warmup):
        flush_buf.zero_()
        step(i)
    fp64_peak = pkg.measure_fp64_peak()

    launches0 = prob.stats()["kernel_launches"]
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kernel_ms = []
    for i in range(args.steps):
        flush_buf.zero_()  # L2 flush between timed iterations (inputs, 50 MB, fit the 126 MB L2)
        ev[i][0].record(stream)
        step(1000 + i)
        ev[i][1].record(stream)
        kernel_ms.append(prob.stats()["last_grid_kernel_ms"])
    barrier()
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "presync_costs.npy"), step.curve.cpu().numpy().astype(np.float64))
    clocks = sampler.stop()
    launches = prob.stats()["kernel_launches"] - launches0
    step_ms = [a.elapsed_time(b) for a, b in ev]
    t = torch.tensor([sum(step_ms) / args.steps, float(np.mean(kernel_ms))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step, kern_ms = float(t[0]), float(t[1])
    value = cells_per_step / (ms_per_step * 1e-3)

    # ---- end to end: host buffers in, curve out, through the C ABI --------------------------
    # N = 1: SetGyroQuaternions + bulk SetTrackResult from host memory, then the grid.  N > 1: the
    # inputs enter through rank 0 only (one validation / staging / PCIe upload instead of N through the
    # same host), its finished device state is replicated to the other ranks over NVLink (NCCL
    # broadcast into the engines' own buffers), then every rank evaluates its offsets.
    e2e_steps = args.steps
    counts = np.full(w.n_frames, w.n_rays)
    st0 = prob.stats()
    bcast_bytes = 0
    marks_on = bool(os.environ.get("RSSYNC_BENCH_MARKS"))
    def e2e_step(call_no):
        m = [time.perf_counter()]
        if rank == 0:
            prob.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
            prob.set_track_batch(w.frame_ids, counts, w.ts_a, w.ts_b, w.rays_a, w.rays_b)
        m.append(time.perf_counter())
        if world > 1:
            sharded.replicate_state(prob, rank=rank, world=world, device=dev)
        m.append(time.perf_counter())
        step(call_no, m)
        if marks_on:
            m.append(time.perf_counter())
            d = np.diff(m) * 1e3
            print(f"[e2e marks] rank {rank} call {call_no}: ingest {d[0]:.2f} replicate {d[1]:.2f} grid {d[2]:.2f} "
                  f"gather {d[3]:.2f} ms", file=sys.stderr, flush=True)

    for c in (1998, 1999):  # untimed warm-up of this path (NCCL sets up its broadcast channels on first use)
        e2e_step(c)
    st0 = prob.stats()
    barrier()
    t0 = time.perf_counter()
    e2e_marks = []
    for i in range(e2e_steps):
        e2e_step(2000 + i)
        e2e_marks.append(time.perf_counter())
    barrier()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    st1 = prob.stats()
    # the curve that came out of the pipelined path (grid behind the ingest / the replication still in
    # flight) against the same call on the now resident state
    e2e_curve = step.curve
    step(2000 + e2e_steps - 1)
    e2e_same = torch.tensor([1.0 if torch.equal(e2e_curve, step.curve) else 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_same, op=dist.ReduceOp.MIN)
    if world > 1:
        ds = prob.device_state()
        bcast_bytes = sum(ds[k][1] for k in ("rays", "orig", "pos", "spline_records")) + w.n_frames * 32
    te = torch.tensor([e2e_s, float(st1["h2d_bytes"] - st0["h2d_bytes"]), float(st1["d2h_bytes"] - st0["d2h_bytes"])],
                      dtype=torch.float64, device=dev)
    if world > 1:
        tm = te.clone()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(te, op=dist.ReduceOp.SUM)
        te[0] = tm[0]
    e2e = {"value": cells_per_step / float(te[0]), "unit": UNIT,
           "h2d_bytes_per_step": int(te[1]) // e2e_steps, "d2h_bytes_per_step": int(te[2]) // e2e_steps,
           "ms_per_step": float(te[0]) * 1e3,
           "what": ("SetGyroQuaternions + SetTrackResult (bulk) from host buffers, grid through the C ABI, curve back on the host"
                    if world == 1 else
                    "rank 0: SetGyroQuaternions + SetTrackResult (bulk) from host buffers; its device state replicated "
                    "to the other ranks by NCCL broadcast over NVLink; every rank's grid slice through the C ABI; "
                    "curve gathered; bytes are summed over ranks"),
           "nvlink_broadcast_bytes_per_step": int(bcast_bytes),
           "equals_resident_state": bool(float(e2e_same[0]) == 1.0),
           "ms_each_step_rank0": [round(1e3 * (b - a), 3) for a, b in zip([t0] + e2e_marks[:-1], e2e_marks)]}

    # ---- roofline of the dominant kernel (presync_kernel) -------------------------------------
    achieved = FLOP_PER_CELL * cells_per_step_rank / (kern_ms * 1e-3) / 1e12
    input_bytes = w.n_frames * ((w.n_rays + 31) // 32 * 32) * 64 + w.quats.shape[0] * 128 + cells_per_step_rank // w.n_rays * 8
    traffic = read_traffic()
    roofline = {"bound": "fp64", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s",
                "frac": achieved / fp64_peak if fp64_peak > 0 else None,
                "peak_source": "measured live: rssync_measure_fp64_peak (dependent DFMA chains, all SMs)",
                "kernel": "presync_kernel", "kernel_ms": kern_ms, "flop_per_cell": FLOP_PER_CELL,
                # dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel on this
                # workload, read from the tracked ncu capture (profiles/presync_traffic.json)
                "traffic": (traffic["dram_bytes_read"] + traffic["dram_bytes_write"])
                if (traffic and w.name == "C2" and hi - lo == OFFSETS_PER_GPU) else None,
                "traffic_source": traffic.get("capture") if traffic else None,
                "exact_estimator_tasks": int(prob.stats()["last_grid_exact_tasks"]),
                "tasks": int(prob.stats()["last_grid_tasks"]),
                "hbm": {"algorithmic_bytes": int(input_bytes),
                        "achieved_gbs": input_bytes / (kern_ms * 1e-3) / 1e9, "peak_gbs": read_peaks().get("hbm_gbs")}}

    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": workload_name(w, n_gpus), "l2": "flushed between timed steps (512 MB memset)",
                      "parallelism": f"offset-sharded x{n_gpus}, inputs replicated"},
           "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline}

    # ---- Sync: syncpoints/s (PreSync on the window + 4 chained Sync, core_testcode.cpp:303-316)
    sync_delays = None
    if not args.no_sync:
        out["sync"], sync_delays = bench_syncpoints(prob, w, "C2: 27 syncpoints (window 60, distance 120)", rank, world,
                                                    barrier, dev, fp64_peak, repeat=3)

    # ---- the sharded configurations north_star names (C3 strong scaling, C4 with 900 syncpoints) --
    if not args.no_scale:
        del flush_buf
        out["scale"] = bench_scale_configs(pkg, sharded, rank, world, barrier, dev, fp64_peak, cores, local_world)

    # ---- the same N GPUs driven by ONE process through the C ABI (rssync_create_multi) -------------
    if world > 1:
        barrier()
        # the other ranks wait on the HOST (the c10d store), not in an NCCL barrier whose spinning
        # kernel would share their GPUs with the run
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            out["one_process_all_gpus"] = bench_in_library_multi(pkg, w, delays, fb, fe, prob, world, args.steps)
            store.set("rssync_in_library_done", "1")
        else:
            store.wait(["rssync_in_library_done"])
        barrier()

    if rank == 0 and not args.no_cpu and world == 1:
        out["cpu_baseline"] = cpu_baseline(w, delays, args.cpu_seconds)
        out["cpu_baseline"]["parity"] = full_size_parity(prob, w, delays, pkg)
        if not args.no_sync:
            out["sync"]["parity"], out["cpu_baseline"]["sync"] = sync_parity_vs_oracle(w, sync_delays)
    elif rank == 0 and not args.no_cpu:
        out["cpu_baseline"] = None
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def bench_in_library_multi(pkg, w, delays, fb, fe, single, n_dev, steps):
    """The headline grid (201 offsets per GPU) through ONE problem spread over all N devices by the
    library itself (rssync_create_multi: what a C++ caller gets with RSSYNC_DEVICES): offsets sharded
    inside the library, one ncclAllGather per call on device buffers.  Run by rank 0 while the other
    ranks wait; the curve is compared bit for bit with the same grid on rank 0's single device."""
    mp = pkg.SyncProblem(seed=100, devices=list(range(n_dev)))
    mp.load(w, bulk=True)
    for i in range(3):
        mp.presync_grid(fb, fe, delays, stream=pkg.STREAM_DEBUG, call_no=i)
    t0 = time.perf_counter()
    for i in range(steps):
        curve = mp.presync_grid(fb, fe, delays, stream=pkg.STREAM_DEBUG, call_no=3000 + i)
    dt = (time.perf_counter() - t0) / steps
    same = bool(np.array_equal(curve, single.presync_grid(fb, fe, delays, stream=pkg.STREAM_DEBUG, call_no=3000 + steps - 1)))
    # end to end: the inputs enter the primary, are replicated by the library (ncclBroadcast), the grid runs
    counts = np.full(w.n_frames, w.n_rays)
    for i in range(-1, 3):  # one untimed pass first (the broadcast channels are set up on first use)
        if i == 0:
            t0 = time.perf_counter()
        mp.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
        mp.set_track_batch(w.frame_ids, counts, w.ts_a, w.ts_b, w.rays_a, w.rays_b)
        e2e_curve = mp.presync_grid(fb, fe, delays, stream=pkg.STREAM_DEBUG, call_no=3000 + steps - 1)
    e2e = (time.perf_counter() - t0) / 3
    same = same and bool(np.array_equal(e2e_curve, curve))  # the pipelined replication delivers the same state
    st = mp.stats()
    cells = len(delays) * w.n_frames * w.n_rays
    res = {"devices": mp.device_count(), "ms_per_step": dt * 1e3, "value": cells / dt, "unit": UNIT,
           "e2e_ms_per_step": e2e * 1e3, "e2e_value": cells / e2e, "equals_one_gpu": same,
           "nccl_calls": int(st["nccl_calls"]), "timing": "wall clock around the C-ABI call (host buffers out)",
           "what": "one process, one rssync_problem over all devices; offsets sharded inside the library, one "
                   "ncclAllGather per call; inputs replicated from the primary by a grouped ncclBroadcast"}
    mp.close()
    return res


def bench_scale_configs(pkg, sharded, rank, world, barrier, dev, fp64_peak, cores, local_world):
    """C3 (10 000 frames x 500 rays x 2001 offsets, strong scaling: offsets sharded) and C4 (30-minute
    trace, a syncpoint every 120 frames = 900 syncpoints, sharded).  The inputs are generated and
    ingested on rank 0 only and replicated to the other GPUs over NVLink; each number is wall time
    including the gather; rank 0 then repeats the whole configuration alone, in the same run on the
    same box, for the speed-up."""
    import torch
    import torch.distributed as dist
    synth = importlib.import_module("rs-sync_b200.synth")
    res = {}

    def problem_for(name, **kw):
        """rank 0 generates + ingests, the others adopt its device state; returns (problem, workload-or-None)"""
        p = pkg.SyncProblem(seed=100)
        w = None
        t0 = time.perf_counter()
        if rank == 0:
            w = synth.make_workload(name, procs=max(1, min(cores, 32)), **kw)
            p.load(w, bulk=True)
            p.flush()
        t_gen = time.perf_counter() - t0
        barrier()
        t0 = time.perf_counter()
        sharded.replicate_state(p, rank=rank, world=world, device=dev)
        barrier()
        return p, w, t_gen, time.perf_counter() - t0

    # ---- C3, strong scaling --------------------------------------------------------------------
    p, w, t_gen, t_rep = problem_for("C3")
    meta = [None]
    if rank == 0:
        meta = [dict(fb=int(w.frame_ids[0]), fe=int(w.frame_ids[-1]) + 1, n_frames=w.n_frames, n_rays=w.n_rays,
                     true_delay=float(w.true_delay[0]))]
    if world > 1:
        dist.broadcast_object_list(meta, src=0)
    m = meta[0]
    delays = np.array([0.0 - 1.0 + 2 * 1.0 * i / 2000 for i in range(2001)])  # core_private.cpp:345
    lo, hi = sharded.shard_range(len(delays), rank, world)
    # warm-up: a few tens of milliseconds of the same grid (the device has idled while rank 0 generated the inputs)
    p.presync_grid(m["fb"], m["fe"], delays[lo:min(hi, lo + 256)], stream=2, call_no=0, offset_index_base=lo)
    each = []
    for _ in range(2):  # twice, the better one counts (both are reported)
        barrier()
        t0 = time.perf_counter()
        curve = sharded.presync_grid_sharded(p, m["fb"], m["fe"], delays, stream=2, call_no=1, rank=rank, world=world, device=dev)
        barrier()
        tt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        each.append(float(tt[0]))
    dt = min(each)
    cells = len(delays) * m["n_frames"] * m["n_rays"]
    c3 = {"config": f"C3: {m['n_frames']} frames x {m['n_rays']} rays x {len(delays)} offsets (radius 1 s, step 1 ms), offsets sharded x{world}",
          "scaling": "strong", "seconds": dt, "cells_per_s": cells / dt,
          "frac_fp64_peak": FLOP_PER_CELL * cells / dt / 1e12 / (fp64_peak * world) if fp64_peak > 0 else None,
          "argmin_delay": float(delays[int(np.argmin(curve))]), "true_delay": m["true_delay"],
          "seconds_each": each, "checksum": float(np.sum(curve)), "synth_seconds_rank0": t_gen, "replicate_seconds": t_rep}
    if world > 1:
        n1, same = None, True
        if rank == 0:
            n1 = None
            for _ in range(2):
                t1 = time.perf_counter()
                whole = p.presync_grid(m["fb"], m["fe"], delays, stream=2, call_no=1)
                n1 = min(n1, time.perf_counter() - t1) if n1 else time.perf_counter() - t1
            same = bool(np.array_equal(whole, curve))
        host_wait(rank, "c3_solo")
        barrier()
        c3.update(n1_seconds_same_run=n1, speedup_vs_one_gpu_same_run=(n1 / dt) if n1 else None, equals_one_gpu=same)
    res["c3_strong"] = c3
    del p, w
    torch.cuda.empty_cache()

    # ---- C4 with 900 syncpoints ------------------------------------------------------------------
    p, w, t_gen, t_rep = problem_for("C4d")
    meta = [None]
    if rank == 0:
        meta = [dict(sps=w.syncpoints(), win=w.sync_window, step=w.presync_step, n_rays=w.n_rays,
                     true=[w.true_delay_at(s) for s in w.syncpoints()], n_frames=w.n_frames,
                     gyro_samples=int(w.quats.shape[0]))]
    if world > 1:
        dist.broadcast_object_list(meta, src=0)
    m = meta[0]

    class Meta:  # what bench_syncpoints needs of a workload
        sync_window, presync_step, n_rays = m["win"], m["step"], m["n_rays"]
        def syncpoints(self): return m["sps"]
        def true_delay_at(self, s): return m["true"][m["sps"].index(s)]
    c4, _ = bench_syncpoints(p, Meta(), f"C4: 30 min 60 fps trace, {len(m['sps'])} syncpoints (window 60, distance 120), "
                             f"{m['n_frames']} tracked frames x {m['n_rays']} rays, {m['gyro_samples']} gyro samples",
                             rank, world, barrier, dev, fp64_peak, repeat=2)
    c4.update(synth_seconds_rank0=t_gen, replicate_seconds=t_rep)
    res["c4_sync"] = c4
    return res


def read_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)
    except Exception:
        return {}


if __name__ == "__main__":
    a = parse()
    # stdout carries the one JSON line and nothing else: libraries that write to file descriptor 1
    # (NCCL prints its version banner there) are sent to stderr for the duration of the run
    sys.stdout.flush()
    _json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = _json_out
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
    _json_out.flush()
