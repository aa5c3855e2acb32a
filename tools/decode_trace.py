#!/usr/bin/env python
"""Host decoder vs device decoder of `himut call`, alternated in one run: per 16 Mb group of the 64 Mb contig of
tools/worker_trace.py (seed 5) and for the 1 Mb BAM of BASELINE configs[0] (synth default seed), the host decode
(hm_bam_read_batch, as the worker calls it) and the device decode (Context.decode_region) split into the copy of the
compressed range, each decode kernel and the read / name round trip; then the worker's BAM -> records wall time with
decode="host", decode="device" and decode="auto".  Bases/s = aligned bases of the decoded reads over the time.  The card's name and
power limit are read in the same run.
--seq: the same for normcounts, which decodes with the 2-bit base stream: host read_batch(seq=True, compact=True) against
decode_region(seq=True), with the device decode without seq timed beside it (k_bam_parse with and without the base
stream), then the normcounts worker's BAM -> tri counts with decode="host", "device" and "auto", whose outputs must agree.
--tags md | md_eqx: the BAMs carry CIGAR + MD:Z instead of cs:Z (the decoders' MD path).
--group S: only the decode group [S, S + GROUP_SPAN) of the 64 Mb contig, no worker runs (A/B of the decode kernels).
    python tools/decode_trace.py [--reps 3] [--seq] [--tags cs] [--group S] [--out profiles/decode_trace_r03.json | decode_trace_norm_r04.json]"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--seq", action="store_true", help="decode with the base stream and time the normcounts worker")
ap.add_argument("--tags", default="cs", choices=["cs", "md", "md_eqx"], help="the alignment tag the BAMs are written with")
ap.add_argument("--group", type=int, default=None, help="time only the decode group starting here, on the 64 Mb contig")
ap.add_argument("--out", default=None)
a = ap.parse_args()
if a.out is None:
    a.out = os.path.join(ROOT, "profiles", "decode_trace_norm_r04.json" if a.seq else "decode_trace_r03.json")

import cases  # noqa: E402
from himut_b200 import bamdec, caller, gtmodel, lib, normcounts, synth, worker  # noqa: E402

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], stdout=subprocess.PIPE, text=True).stdout
tmp = tempfile.mkdtemp()
inputs, refs = {}, {}
for label, n, seed in (("64mb", 64_000_000, 5), ("1mb", 1_000_000, None))[:1 if a.group is not None else 2]:
    d = synth.generate(n, **({"seed": seed} if seed is not None else {}), copy=False)
    path = os.path.join(tmp, label + ".bam")
    bamdec.write_batch_bam(path, "chr1", n, d.batch, **({"tags": a.tags} if a.tags != "cs" else {}))
    inputs[label] = (path, n, os.path.getsize(path))
    if a.seq:
        refs[path] = bytes(d.ref)
    del d
G = worker.GROUP_SPAN


def groups(n):
    """the worker's decode groups, then (64 Mb contig) smaller regions at its start: where the two decoders cross"""
    if a.group is not None:
        return [(a.group, min(a.group + G, n))]
    g = [(s, min(s + G, n)) for s in range(0, n, G)]
    return g + [(0, L) for L in (1_000_000, 2_000_000, 4_000_000, 8_000_000) if L < n]


def host_decode(nb, s, e, seq=False):
    t0 = time.perf_counter()
    b, _cq = nb.read_batch("chr1", s, e, copy=False, seq=seq, compact=True)
    return time.perf_counter() - t0, b.n_reads


def device_decode(ctx, nb, s, e, seq=False):
    t0 = time.perf_counter()
    r = ctx.decode_region(nb, "chr1", s, e, seq=seq)
    wall = time.perf_counter() - t0
    ab = ctx.read_back().aligned_bases
    return wall, r.n_reads, dict(ctx.last_decode_times), ab


g = gtmodel.DEFAULT_CALL_ARGS


def worker_run(path, n, mode):
    real = caller.call_region
    caller.call_region = lambda *x, **k: real(*x, **dict(k, decode=mode))
    try:
        lst, log = {}, {}
        t0 = time.perf_counter()
        caller.get_somatic_substitutions(
            "chr1", path, None, None, [("chr1", s, e) for s, e in cases.chunkloci(0, n)], {}, {}, {}, g["min_qv"], g["min_mapq"],
            g["qlen_lower_limit"], g["qlen_upper_limit"], g["min_sequence_identity"], g["min_gq"], g["min_bq"], g["min_trim"],
            g["max_mismatch_count"], g["mismatch_window"], g["md_threshold"], g["min_ref_count"], g["min_alt_count"],
            g["min_hap_count"], 1e-6, g["germline_snv_prior"], 1e-4, False, True, False, lst, log)
        return time.perf_counter() - t0, len(lst["chr1"]), list(log["chr1"])
    finally:
        caller.call_region = real


def norm_worker_run(path, n, mode):
    real = normcounts.normcounts_region
    normcounts.normcounts_region = lambda *x, **k: real(*x, **dict(k, decode=mode))
    try:
        ccs, rt, log = {}, {}, {}
        t0 = time.perf_counter()
        ties = normcounts.get_callable_tricounts(
            "chr1", refs[path], path, None, None, [("chr1", s, e) for s, e in cases.chunkloci(0, n)], {}, {}, {}, g["min_qv"],
            g["min_mapq"], g["min_trim"], g["qlen_lower_limit"], g["qlen_upper_limit"], g["min_sequence_identity"], g["min_gq"],
            g["min_bq"], g["mismatch_window"], g["max_mismatch_count"], g["min_ref_count"], g["min_alt_count"], g["min_hap_count"],
            float(g["md_threshold"]), 1e-6, g["germline_snv_prior"], 1e-4, False, False, ccs, rt, log)
        return time.perf_counter() - t0, sum(ccs["chr1"].values()), (ccs["chr1"], rt["chr1"], list(log["chr1"]), ties)
    finally:
        normcounts.normcounts_region = real


out = {"card": card.strip(), "tags": a.tags, "group_span": G, "threads_host_decoder": bamdec.default_threads(), "inputs": {}, "decode": [], "worker": []}
if a.seq:
    out["seq"] = True
    out["device_decode_min_bytes"] = {"call": caller.DEVICE_DECODE_MIN_BYTES, "normcounts": normcounts.DEVICE_DECODE_MIN_BYTES}
ctx = lib.Context(0)
for label, (path, n, size) in inputs.items():
    out["inputs"][label] = {"contig_len": n, "bam_bytes": size}
    nb = bamdec.NativeBam(path)
    for s, e in groups(n):  # warm-up of every shape (module load, allocations)
        host_decode(nb, s, e, a.seq)
        device_decode(ctx, nb, s, e, a.seq)
        if a.seq:
            device_decode(ctx, nb, s, e)
    for rep in range(a.reps):
        for s, e in groups(n):
            th, nh = host_decode(nb, s, e, a.seq)
            td, nd, kt, ab = device_decode(ctx, nb, s, e, a.seq)
            assert nh == nd
            pl = nb.plan("chr1", s, e)
            row = {"input": label, "rep": rep, "start": s, "end": e, "reads": nd, "aligned_bases": ab,
                   "compressed_bytes": int(pl.comp_bytes), "host_s": th, "device_s": td, "device_ms": kt,
                   "host_bases_per_s": ab / th, "device_bases_per_s": ab / td}
            if a.seq:  # the same region without the base stream, right after: k_bam_parse with and without it
                row["device_noseq_s"], _, row["device_noseq_ms"], _ = device_decode(ctx, nb, s, e)
            out["decode"].append(row)
            print("%s [%d, %d) %.0f MB rep %d: host %.1f ms, device %.1f ms %s" % (label, s, e, pl.comp_bytes / 1e6, rep, th * 1e3,
                                                                                     td * 1e3, {k: round(v, 2) for k, v in kt.items()}),
                  file=sys.stderr)
    nb.close()
    if a.group is not None:
        continue
    nb = bamdec.NativeBam(path)
    whole_bases = nb.read_batch("chr1", 0, n, seq=False).aligned_bases
    nb.close()
    run = norm_worker_run if a.seq else worker_run
    for mode in ("host", "device", "auto"):  # warm-up
        run(path, n, mode)
    ref = None
    for rep in range(a.reps):
        for mode in ("host", "device", "auto"):
            t, rows, log = run(path, n, mode)
            ref = ref or (rows, log)
            assert (rows, log) == ref, "the two decode paths give different %s" % ("tri counts" if a.seq else "records")
            out["worker"].append({"input": label, "rep": rep, "decode": mode, "wall_s": t, "callable_tri" if a.seq else "rows": rows,
                                  "aligned_bases": whole_bases, "bases_per_s": whole_bases / t})
            print("%s worker decode=%s rep %d: %.3f s (%d rows)" % (label, mode, rep, t, rows), file=sys.stderr)
ctx.close()
os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as f:
    json.dump(out, f, indent=1)
print(json.dumps({k: v for k, v in out.items() if k in ("card",)}))
