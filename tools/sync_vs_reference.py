"""Characterises how far the engine's arithmetic contract ("spec": DESIGN.md §3) moves Sync's
result away from the reference's own arithmetic.

Sync's delay gradient is a central difference with h = 1e-6 s of a sum of ~1e3..1e4
(core_private.cpp:96-97,112), so the last-bit differences between two correct evaluations of the
loss (FMA placement, summation order, log1p) are amplified by 1/(2h) and — because the loop stops
on six consecutive steps below 1e-4 (:316-324) — can leave it on a different iteration.  This script
measures that on many windows:

    spec oracle  (oracle/rssync_oracle.cpp, the arithmetic the CUDA engine reproduces bit for bit,
                  tests/test_gpu_parity.py)
    reference    (oracle/_ref/librssync_ref.so: the unmodified reference sources compiled here
                  against oracle/shim; needs /root/reference at BUILD time only)

and, as the yardstick, a SECOND build of the same unmodified reference sources in which the compiler
may contract a*b+c into FMAs (oracle/_ref/librssync_ref_fma.so, `make -C oracle ref_fma`; what a
-march=native release build does).  It writes the distributions of |delay_spec - delay_ref| and of
|delay_ref_fma - delay_ref| to profiles/: the second one is how far the reference moves away from
ITSELF under an equally valid rounding of the same expressions.  CPU only.  The windows' recorded
results also go to tests/golden/sync_reference.json, which the test suite replays where the
reference is not at hand (tests/recorded_reference.py).

usage: python tools/sync_vs_reference.py [--windows 56] [--out profiles/r02_sync_vs_reference.json]
                                         [--golden tests/golden/sync_reference.json]
"""
import argparse
import importlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=56)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r02_sync_vs_reference.json"))
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 1)
    ap.add_argument("--golden", default=os.path.join(ROOT, "tests", "golden", "sync_reference.json"))
    a = ap.parse_args()
    from oracle import loader, ref_loader
    if not ref_loader.available():
        raise SystemExit("oracle/_ref/librssync_ref.so is missing: run `make -C oracle ref` where /root/reference exists")
    synth = importlib.import_module("rs-sync_b200.synth")
    rows = []
    fma_path = os.path.join(ROOT, "oracle", "_ref", "librssync_ref_fma.so")
    if not os.path.exists(fma_path):
        fma_path = None
    t_begin = time.time()
    # C1-shaped data (300 frames x 100 rays, 1 kHz gyro), several world seeds / noise levels, windows
    # of 24 and 60 frames (core_testcode's sync_window), starting delays one PreSync step around the
    # true delay, 1-2 chained Sync calls (core_testcode.cpp:314 chains four)
    scenes = [dict(seed=1), dict(seed=2), dict(seed=3, noise_px=0.6), dict(seed=4, outlier_frac=0.2),
              dict(seed=5, true_delay=-0.021), dict(seed=6), dict(seed=7, noise_px=0.15)]
    per_scene = (a.windows + len(scenes) - 1) // len(scenes)
    for si, kw in enumerate(scenes):
        w = synth.make_workload("C1", **kw)
        o = loader.OracleProblem(threads=a.threads, seed=100).load(w)
        r = ref_loader.RefProblem(threads=a.threads, seed=100).load(w)
        r2 = ref_loader.RefProblem(threads=a.threads, seed=100, lib_path=fma_path).load(w) if fma_path else None
        td = float(w.true_delay[0])
        for k in range(per_scene):
            if len(rows) >= a.windows:
                break
            win = 60 if k % 2 == 0 else 24
            fb = int(w.frame_ids[0]) + (k * 29) % (w.n_frames - win - 1)
            start = td + (0.002 if k % 3 == 0 else -0.0013 if k % 3 == 1 else 0.0004)
            call = 10 * k + 3
            o.set_rng(100, call)
            r.set_rng(100, call)
            if r2:
                r2.set_rng(100, call)
            do = dr = dr2 = start
            chain = 2 if k % 4 == 0 else 1
            for _ in range(chain):
                co, do = o.Sync(do, fb, fb + win, td, 0.2)
                cr, dr = r.Sync(dr, fb, fb + win, td, 0.2)
                if r2:
                    _, dr2 = r2.Sync(dr2, fb, fb + win, td, 0.2)
            rows.append(dict(scene=si, workload=kw, call_no=call, frames=win + 1, first_frame=fb, start=start, chain=chain,
                             delay_spec=do, delay_ref=dr, cost_spec=co, cost_ref=cr,
                             abs_delay_diff=abs(do - dr), rel_cost_diff=abs(co - cr) / abs(cr),
                             delay_ref_fma=dr2 if r2 else None,
                             abs_delay_diff_ref_vs_ref_fma=abs(dr2 - dr) if r2 else None))
            print(f"[{len(rows):3d}/{a.windows}] scene {si} fb {fb} win {win} chain {chain}: "
                  f"|d_spec - d_ref| = {abs(do - dr):.3e}  |d_ref_fma - d_ref| = {abs(dr2 - dr) if r2 else float('nan'):.3e}",
                  file=sys.stderr, flush=True)
    d = np.array([x["abs_delay_diff"] for x in rows])
    c = np.array([x["rel_cost_diff"] for x in rows])
    summary = dict(
        what="|Sync delay (spec arithmetic = CUDA engine) - Sync delay (unmodified reference sources, oracle/_ref)|, seconds",
        windows=len(rows), max_abs_delay_diff=float(d.max()), median_abs_delay_diff=float(np.median(d)),
        p90_abs_delay_diff=float(np.quantile(d, 0.9)),
        frac_within_1e_9=float(np.mean(d <= 1e-9)), frac_within_1e_6=float(np.mean(d <= 1e-6)),
        frac_within_1e_5=float(np.mean(d <= 1e-5)), frac_within_1e_4=float(np.mean(d <= 1e-4)),
        max_rel_cost_diff=float(c.max()), median_rel_cost_diff=float(np.median(c)),
        reference_stop_threshold_s=1e-4, seconds=time.time() - t_begin, threads=a.threads)
    if fma_path:
        e = np.array([x["abs_delay_diff_ref_vs_ref_fma"] for x in rows])
        summary["reference_vs_its_own_fma_build"] = dict(
            what="|Sync delay (reference, -ffp-contract=fast -mfma) - Sync delay (reference, -ffp-contract=off)|, same windows",
            max_abs_delay_diff=float(e.max()), median_abs_delay_diff=float(np.median(e)),
            p90_abs_delay_diff=float(np.quantile(e, 0.9)), frac_within_1e_9=float(np.mean(e <= 1e-9)),
            frac_within_1e_6=float(np.mean(e <= 1e-6)), frac_within_1e_4=float(np.mean(e <= 1e-4)))
    with open(a.out, "w") as f:
        json.dump(dict(summary=summary, rows=rows), f, indent=1)
    write_golden(rows, a.golden)
    print(json.dumps(summary, indent=1))


def write_golden(rows, path):
    """the replayable part of `rows` (workload arguments, window, start, chain, call number and both
    results, floats as hex) in the format tests/recorded_reference.py reads"""
    comment = ("Sync results of the unmodified rs-sync reference sources (compiled with -ffp-contract=off "
               "against oracle/shim) and of the spec oracle, recorded by tools/sync_vs_reference.py "
               "(profiles/r02_sync_vs_reference.json).  Each row: w = synth.make_workload('C1', **workload); "
               "problem loaded with seed 100; set_rng(100, call_no); d = start; `chain` times "
               "(cost, d) = Sync(d, frame_begin, frame_end, w.true_delay[0], 0.2).")
    out = []
    for r in rows:
        h = lambda k: float(r[k]).hex()
        out.append({"workload": r["workload"], "frame_begin": r["first_frame"],
                    "frame_end": r["first_frame"] + r["frames"] - 1, "start_hex": h("start"), "chain": r["chain"],
                    "call_no": r["call_no"], "delay_ref_hex": h("delay_ref"), "cost_ref_hex": h("cost_ref"),
                    "delay_spec_hex": h("delay_spec"), "cost_spec_hex": h("cost_spec")})
    with open(path, "w") as f:
        f.write('{"comment": ' + json.dumps(comment) + ',\n "rows": [\n')
        f.write(",\n".join("  " + json.dumps(r) for r in out))
        f.write("\n ]}\n")


if __name__ == "__main__":
    main()
