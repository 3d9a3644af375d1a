"""Sync results of the unmodified rs-sync reference recorded beside the spec oracle's
(tests/golden/sync_reference.json, written by tools/sync_vs_reference.py): lets the oracle and the
engine be compared with the reference where its sources are not at hand."""
import json
import os

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sync_reference.json")

# |Sync delay (spec) - Sync delay (reference)| over the 56 recorded windows: at most 3.8e-4 s (93% within
# the reference's stopping threshold of 1e-4 s); a second build of the reference itself with FMA
# contraction moves its own delay by up to 2.7e-4 s on the same windows
DELAY_BOUND = 4e-4


def rows():
    """one dict per window: workload (synth.make_workload('C1', **workload)), frame_begin, frame_end,
    start, chain, call_no and the recorded delay_ref, cost_ref, delay_spec, cost_spec"""
    with open(PATH) as f:
        g = json.load(f)
    h = float.fromhex
    return [dict(r, start=h(r["start_hex"]), delay_ref=h(r["delay_ref_hex"]), cost_ref=h(r["cost_ref_hex"]),
                 delay_spec=h(r["delay_spec_hex"]), cost_spec=h(r["cost_spec_hex"])) for r in g["rows"]]


def replay(make_problem, workload):
    """run every recorded window on problems from make_problem(w); yields (row, cost, delay)"""
    problems = {}
    for r in rows():
        key = json.dumps(r["workload"], sort_keys=True)
        if key not in problems:
            w = workload("C1", **r["workload"])
            problems[key] = (w, make_problem(w))
        w, p = problems[key]
        p.set_rng(100, r["call_no"])
        d = r["start"]
        for _ in range(r["chain"]):
            c, d = p.Sync(d, r["frame_begin"], r["frame_end"], float(w.true_delay[0]), 0.2)
        yield r, c, d
