#!/usr/bin/env python
"""Cost of the callable-base track of `himut normcounts` (HM_OPT_CALLABLE_TRACK) on the 64 Mb, 30x contig of bench.py
(synth seed 20260101, 320 chunks of 200 kb, resident batch uploaded as the worker uploads it): normcounts_chunks with
the track off and on, alternated, each timed with CUDA events over --steps calls; then one call of each with the
kernel events on (hm_last_kernel_times) for the extra kernel time, and the runs: how many, the bytes
hm_last_callable_runs copies back and the time of that copy.  The card's name and power limit are read in the same
run.  Results must agree: the tallies of both arms are compared, and the runs summed per bin against them.
    python tools/callable_trace.py [--steps 10] [--reps 3] [--out profiles/callable_trace_r08.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=10)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--contig-mb", type=int, default=64)
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "callable_trace_r08.json"))
a = ap.parse_args()

import numpy as np  # noqa: E402
import torch  # noqa: E402

import __graft_entry__ as g  # noqa: E402

g.build()
import cases  # noqa: E402
from himut_b200 import bamdec, gtmodel, lib, synth  # noqa: E402
from test_callable_track import run_sums, tri_bins  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


n = a.contig_mb * 1_000_000
d = synth.generate(n, seed=20260101, copy=False)
chunks = d.batch.chunk_table(cases.chunkloci(0, n))
ctx = lib.Context(0)
ctx.set_params(gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS))
ctx.set_site_sets()
ctx.upload_compact(d.batch, bamdec.compact_bq(d.batch))
ctx.set_reference(d.ref)
stream = torch.cuda.Stream()
ctx.set_stream(stream.cuda_stream)


def timed(on):
    ctx.callable_track(on)
    ctx.kernel_timing(False)
    ctx.normcounts_chunks(None, chunks)  # warm: buffers sized, modules loaded
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(a.steps):
        r = ctx.normcounts_chunks(None, chunks)
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1) / a.steps, r


ms = {"off": [], "on": []}
res = {}
for _ in range(a.reps):
    for arm in ("off", "on"):
        t, res[arm] = timed(arm == "on")
        ms[arm].append(t)
same = all(np.array_equal(np.asarray(x), np.asarray(y)) for x, y in zip(res["off"][:3], res["on"][:3])) and res["off"][3] == res["on"][3]

kern = {}
for arm in ("off", "on"):
    ctx.callable_track(arm == "on")
    ctx.kernel_timing(True)
    ctx.normcounts_chunks(None, chunks)
    kern[arm] = ctx.last_kernel_times()
t0 = time.perf_counter()
runs = ctx.last_callable_runs()
copy_ms = (time.perf_counter() - t0) * 1e3
ctx.callable_track(False)
r_ref, r_ccs, total = run_sums(runs, tri_bins(d.ref))
sums_ok = bool(np.array_equal(r_ref, res["on"][1]) and np.array_equal(r_ccs, res["on"][0]) and total == int(res["on"][2][13]))

k_off, k_on = sum(v for _k, v in kern["off"]), sum(v for _k, v in kern["on"])
out = {
    "card": card(), "contig_bases": n, "chunks": int(len(chunks)), "depth": 30, "steps": a.steps, "reps": a.reps,
    "ms_per_call_off": ms["off"], "ms_per_call_on": ms["on"],
    "median_extra_ms_per_call": float(np.median(ms["on"]) - np.median(ms["off"])),
    "kernel_ms_off": kern["off"], "kernel_ms_on": kern["on"], "extra_kernel_ms": k_on - k_off,
    "track_kernels_ms": {k: v for k, v in kern["on"] if k in ("k_track_count", "k_track_emit")},
    "runs": int(runs.size), "counted_positions": int(r_ref.sum()), "positions_per_run": float(r_ref.sum() / max(runs.size, 1)),
    "bytes_copied_back": int(runs.nbytes), "copy_ms_host_clock": copy_ms,
    "device_track_bytes": int(4 * sum(((int(e) - int(s) + 31) // 32) * 32 for s, e in zip(chunks["start"], chunks["end"]))),
    "tallies_identical_on_off": bool(same), "runs_sum_to_tallies": sums_ok,
}
os.makedirs(os.path.dirname(a.out), exist_ok=True)
with open(a.out, "w") as f:
    json.dump(out, f, indent=1)
print(json.dumps({k: v for k, v in out.items() if k not in ("kernel_ms_off", "kernel_ms_on")}))
ctx.close()
