#!/usr/bin/env python
"""bench.py — `himut call` hot-path throughput on synthetic 30x CCS data (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--contig-mb M] [--genome-mb G] [--dump-outputs DIR]

--dump-outputs DIR (N = 1, --impl ours only): the records and counters of the headline call's last timed step as .npy.

A step is one pass of the whole `himut call` device path (k_call_pairs -> k_site_sort -> k_call_scan -> k_site_reduce,
one host synchronisation, host som_seen replay) over the workload's packed read batches.

N = 1 (the driver's BENCH run): BASELINE configs[1], one 64 Mb contig at 30x.
  value   aligned CCS bases/s with the batch already resident in HBM (hm_call_chunks), CUDA events on the launching
          stream, barrier + synchronize on both sides
  e2e     the same metric through the C-ABI call the worker mirrors make (himut_b200/caller.py: hm_upload_batch_compact
          + hm_call_chunks = hm_call_batch_compact) with HOST buffers exactly as the native BAM decoder leaves them
          (the contig is written to a BAM and decoded back, outside the timed region): pinned host -> device copies,
          quality expansion, the whole path and the records back, all inside the timed region
  bam_to_vcf  BAM on disk (page cache) -> VCF on disk through the worker mirror itself (decode included)
  roofline  dominant kernel (k_call_scan) against the measured HBM copy bandwidth, and the whole step (`frac_step`)
  genome  BASELINE configs[2] scaled to --genome-mb: 24 contigs with human length ratios, chunk runs sharded by
          himut_b200.genome.plan_runs — on one GPU here, so that the N > 1 lines have their strong-scaling base
  cpu_baseline  the CPU oracle port on the host cores, a bounded sample of the same contig
N > 1 (torchrun, one rank per GPU): the genome workload is the headline, STRONG scaling: the same genome for every N,
  chunk runs of long contigs on different GPUs, no data-path collective (the 15 log counters are all-reduced over
  NCCL); value = the genome's aligned bases x steps / the slowest rank's time; `imbalance` = max / mean bases per rank.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

METRIC = "aligned CCS bases/sec (himut call, 30x synthetic)"
DUMP_BYTES = 64 << 20  # --dump-outputs: at most this much in all
# chr1 .. chr22, X, Y in Mb (GRCh38, rounded): the length ratios of BASELINE configs[2]'s 3.1 Gb genome
HUMAN_MB = [248, 242, 198, 190, 181, 171, 159, 145, 138, 133, 135, 133, 114, 107, 102, 90, 83, 80, 58, 64, 46, 50, 156, 57]


def chunkloci(end):
    out = [(1, 200000)]
    starts = list(range(200000, end, 200000))
    for i, s in enumerate(starts[:-1]):
        out.append((s, starts[i + 1]))
    out.append((starts[-1], end - 2))
    return out


def make_workload(contig_len, seed):
    from himut_b200 import gtmodel, synth
    d = synth.generate(contig_len, seed=seed, copy=False)
    params = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
    chunks = d.batch.chunk_table(chunkloci(contig_len))
    return d, params, chunks


def batch_counts(batch):
    return int(batch.qlen.astype(np.int64).sum()), int(batch.ops.size), int(batch.n_reads)


def scan_alg_bytes(batch):
    """algorithmic bytes of one k_call_scan launch (DESIGN.md §4): every quality byte once, every op word once (the
    prefix scan is redone in registers), 40 B of per-read metadata; the entries it writes (4 B per (site, covering
    read)) are left out, so the figure is a lower bound of what the kernel must move"""
    n_base, n_op, n_read = batch_counts(batch)
    return 1.0 * n_base + 4.0 * n_op + 40.0 * n_read


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(suffix=".csv")
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.proc.wait()
        self.f.close()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            p = [x.strip() for x in line.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(gpu_index):
    """one process per GPU: run it on the cores next to that GPU (NVML's ideal CPU set), so eight ranks do not
    share cores or cross sockets for their pinned-memory copies"""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        allowed = os.sched_getaffinity(0)
        if cpus & allowed:
            os.sched_setaffinity(0, cpus & allowed)
    except Exception:
        pass


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(alg_bytes):
    """DRAM bytes per k_call_scan launch: the dram / algorithmic ratio of the committed `ncu --set full` capture
    (profiles/traffic.json, 64 Mb contig) applied to this launch's algorithmic bytes — not measured in this run"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return float(json.load(open(p))["k_call_scan_dram_over_alg"]) * alg_bytes
    except Exception:
        return None


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_baseline(d, params, chunks, n_chunks, threads=1):
    """oracle port on `threads` host threads, each over its own run of n_chunks consecutive chunks of the contig
    (the reference's own parallelism is one worker per contig, caller.py:766-810: a thread here stands for one such
    worker; ctypes drops the GIL for the duration of the C call) -> (bases/s, bases, seconds, threads used)"""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle
    b = d.batch
    threads = max(1, min(threads, len(chunks) // max(1, n_chunks)))
    groups = [chunks[t * n_chunks:(t + 1) * n_chunks] for t in range(threads)]
    kind, val = b.ops & 3, (b.ops >> 2).astype(np.int64)
    qspan = np.where(kind == 0, val, 0) + (kind == 1) + np.where(kind == 2, val, 0)
    per_read = np.add.reduceat(qspan, b.op_off.astype(np.int64))
    bases = 0
    for sub in groups:
        lo, hi = int(sub["read_lo"].min()), int(sub["read_hi"].max())
        ov = (b.tstart[lo:hi] < int(sub["end"][-1])) & (b.tend[lo:hi] > int(sub["start"][0]))
        bases += int(per_read[lo:hi][ov].sum())
    cap = max(4096, int(b.ops.size) // max(1, len(chunks)) * n_chunks * 4)
    t0 = time.perf_counter()
    if threads == 1:
        oracle.call_chunks(params, b, groups[0], cap=cap)
    else:
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(lambda sub: oracle.call_chunks(params, b, sub, cap=cap), groups))
    dt = time.perf_counter() - t0
    return bases / dt, bases, dt, threads


PY_REF_NOTE = ("the reference itself is pure Python and its I/O dependencies (pysam, natsort, pytabix) are not on this box: the arm times "
               "oracle/himut_oracle.c, a C restatement pinned to the reference's outputs (tests/golden); the unmodified Python "
               "reference ran at 5.0e5 (`call`) and 1.5e5 (`normcounts`) aligned bases/s on one core of the build container "
               "(tests/golden/*_config0_1mb.json: reference_seconds), i.e. the C port is ~300x faster per core than what it stands for")


def run_reference(args, rank, world):
    """--impl reference: the CPU implementation of the path, one thread per host core, on a bounded sample of the
    N = 1 workload.  Nothing of the product is loaded: only the oracle library and the data generator."""
    if rank != 0:
        return
    contig_len = args.contig_mb * 1_000_000
    d, params, chunks = make_workload(contig_len, args.seed)
    threads = host_threads()
    n = max(1, min(len(chunks) // threads, args.cpu_chunks))
    for _ in range(args.warmup):
        cpu_baseline(d, params, chunks, n, threads)
    tot, el = 0, 0.0
    for _ in range(args.steps):
        v, bases, dt, used = cpu_baseline(d, params, chunks, n, threads)
        tot += bases
        el += dt
    value = tot / el
    sample = "%d threads x %d consecutive chunks = %d of %d chunks (%.1f Mb, %d aligned bases) of the %d Mb 30x contig per step" % (
        used, n, used * n, len(chunks), used * n * 0.2, bases, args.contig_mb)
    loaded = [ln.split()[-1] for ln in open("/proc/self/maps") if "libhimut" in ln and ln.rstrip().endswith(".so")]
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "bases/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/f64", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": value, "unit": "bases/s", "cores": used, "kind": "port", "sample": sample, "note": PY_REF_NOTE},
        "e2e": {"value": value, "unit": "bases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "native_libraries_mapped": sorted(set(os.path.basename(p) for p in loaded)),
    }))


def workload_config(args, world):
    if world == 1:
        return {"workload": "himut call on a %d Mb synthetic contig at 30x CCS (15 kb reads, cs tags), %d x 200 kb chunks"
                            % (args.contig_mb, len(chunkloci(args.contig_mb * 1_000_000))),
                "baseline_config": "configs[1]" if args.contig_mb == 64 else "custom",
                "contig_mb": args.contig_mb, "depth": 30, "parallelism": "one GPU",
                "l2": "inputs (>= 2 GB per step) are larger than the 126 MB L2; no explicit flush"}
    return {"workload": "himut call on a %d Mb synthetic genome at 30x CCS: 24 contigs with the length ratios of GRCh38 (BASELINE "
                        "configs[2] at 1/%.0f scale: the 3.1 Gb genome is 116 GB of packed reads and cannot be generated inside the "
                        "bench's time budget), 200 kb chunks, chunk runs sharded over %d GPUs by himut_b200.genome.plan_runs"
                        % (args.genome_mb, 3100.0 / args.genome_mb, world),
            "baseline_config": "configs[2] (scaled)", "genome_mb": args.genome_mb, "depth": 30,
            "parallelism": "chunk runs, contiguous equal-weight partition x%d" % world,
            "l2": "every rank's inputs are larger than the 126 MB L2; no explicit flush"}


# ------------------------------------------------------------------------------------------------ helpers
def slice_batch(batch, lo, hi):
    """reads [lo, hi) of a batch as a batch of their own (array views, offsets rebased); without a base stream"""
    from himut_b200 import abi
    if hi <= lo:
        lo = hi = 0
    b0 = int(batch.bq_off[lo]) if hi > lo else 0
    b1 = (int(batch.bq_off[hi - 1]) + ((int(batch.qlen[hi - 1]) + 15) & ~15)) if hi > lo else 16
    o0 = int(batch.op_off[lo]) if hi > lo else 0
    o1 = (int(batch.op_off[hi - 1]) + int(batch.n_ops[hi - 1])) if hi > lo else 0
    skip = ("seq", "bq", "ops", "seq_off", "bq_off", "op_off")
    kw = {name: getattr(batch, name)[lo:hi] for name, _ in abi.ReadBatch._FIELDS if name not in skip}
    kw["bq_off"] = batch.bq_off[lo:hi] - np.uint64(b0)
    kw["op_off"] = batch.op_off[lo:hi] - np.uint64(o0)
    kw["bq"], kw["ops"] = batch.bq[b0:b1], batch.ops[o0:o1]
    kw["seq"], kw["seq_off"] = np.zeros(0, np.uint8), np.zeros(0, np.uint64)
    return abi.ReadBatch(keepalive=batch, **kw)


def aligned_per_read(batch):
    kind, val = batch.ops & 3, (batch.ops >> 2).astype(np.int64)
    qspan = np.where(kind == 0, val, 0) + (kind == 1) + np.where(kind == 2, val, 0)
    return np.add.reduceat(qspan, batch.op_off.astype(np.int64)) if batch.n_reads else np.zeros(0, np.int64)


class Timer:
    """CUDA events on the launching stream, barrier + synchronize on both sides"""

    def __init__(self, torch, dist, world, stream):
        self.torch, self.dist, self.world, self.stream = torch, dist, world, stream

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def run(self, fn, steps, after=None, streams=()):
        """streams: the CUDA streams the timed work is launched on when it is not the bench's own (contexts with a stream
        each): they wait for the opening event and the closing event waits for them, so the two events bracket the work
        on the device whatever stream it ran on"""
        self.barrier()
        e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for st in streams:
            st.wait_event(e0)
        for _ in range(steps):
            fn()
        if after:
            after()
        for st in streams:
            ev = self.torch.cuda.Event()
            ev.record(st)
            self.stream.wait_event(ev)
        e1.record(self.stream)
        self.barrier()
        return e0.elapsed_time(e1)


def dump_outputs(path, rec, log):
    """the site records and the 15 log counters a call returns, as DIR/records_<field>.npy and DIR/log.npy in float64
    (every field is an integer that float64 holds exactly).  The device returns records in no particular order: they
    are sorted on all their fields first, so that two builds can be compared array for array.  Past DUMP_BYTES, the
    records whose (chunk, tpos, ref, alt) hash lowest are written: the choice depends on each record's key alone, so
    two builds whose record sets differ in a few sites still write the same sample apart from those sites."""
    os.makedirs(path, exist_ok=True)
    rec = np.sort(rec, order=["chunk", "tpos", "ref", "alt"])  # the fields not named break the ties
    fields = [n for n in rec.dtype.names if n != "pad0"]
    row_bytes = 8 * sum(int(np.prod(rec.dtype[n].shape)) for n in fields)
    cap = (DUMP_BYTES - (1 << 20)) // row_bytes  # 1 MB for the counters and the .npy headers
    if rec.size > cap:
        u = np.uint64
        h = (rec["chunk"].astype(u) << u(40)) ^ (rec["tpos"].astype(u) << u(8)) ^ (rec["ref"].astype(u) << u(4)) ^ rec["alt"].astype(u)
        for shift, mul in ((30, 0xBF58476D1CE4E5B9), (27, 0x94D049BB133111EB)):  # splitmix64 finaliser
            h = (h ^ (h >> u(shift))) * u(mul)
        h ^= h >> u(31)
        rec = rec[np.sort(np.lexsort((np.arange(rec.size), h))[:cap])]
    for n in fields:
        np.save(os.path.join(path, "records_%s.npy" % n), rec[n].astype(np.float64))
    np.save(os.path.join(path, "log.npy"), np.asarray(log, np.float64))


def kernel_breakdown(ctx, fn, reps=3):
    """per-kernel CUDA-event times and the launch count of a call, measured outside the timed loops"""
    ctx.kernel_timing(True)
    acc, launches = {}, 0
    for _ in range(reps):
        fn()
        for name, ms in ctx.last_kernel_times():
            acc.setdefault(name, []).append(ms)
        launches = ctx.last_timing()[1]
    ctx.kernel_timing(False)
    return {k: float(np.mean(v)) for k, v in acc.items()}, launches


# ------------------------------------------------------------------------------------------------ N = 1: configs[1]
def leg_contig(args, T, ctx, d, params, chunks, tmpdir):
    """the 64 Mb contig on one GPU: resident, end to end from the decoder's buffers, kernel breakdown"""
    from himut_b200 import bamdec
    batch = d.batch
    aligned = d.aligned_bases
    ctx.set_params(params)
    ctx.set_site_sets()
    ctx.omit_restatements(True)  # germline restatements are counted on the device and not copied back (caller.py:338-345)
    ctx.kernel_timing(False)
    # ---- resident ----
    # As the worker drives the device (himut_b200/caller.py:call_region): two contexts of the process alternate from
    # call to call, the next call is enqueued before the previous one is collected, so the device goes from one to the
    # other without waiting for the host.  Both hold the batch; each has a stream of its own.
    from himut_b200 import lib as _lib
    ctx_b = _lib.Context(ctx.device)
    pair, streams = [ctx, ctx_b], [T.torch.cuda.Stream(), T.torch.cuda.Stream()]
    for c, st in zip(pair, streams):
        c.set_stream(st.cuda_stream)
        c.set_params(params)
        c.set_site_sets()
        c.omit_restatements(True)
        c.kernel_timing(False)
        c.upload(batch.without_seq())
    state = {"k": 0, "pending": None}

    def step():
        c = pair[state["k"] % 2]
        state["k"] += 1
        c.call_chunks_submit(chunks)
        if state["pending"] is not None:
            state["rec"], state["log"] = state["pending"].call_chunks_collect(view=True)
        state["pending"] = c

    def drain():
        if state["pending"] is not None:
            state["rec"], state["log"] = state["pending"].call_chunks_collect(view=True)
            state["pending"] = None
        for c in pair:
            c.records_wait()

    for _ in range(2 * args.warmup + 4):  # each context sizes and page-locks its two record buffers in its first calls
        step()
    drain()
    ms_total = T.run(step, args.steps, after=drain, streams=streams)
    rec, log = state["rec"].copy(), state["log"]
    assert ctx.last_call_path() == 2, "the fused device path did not run"
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rec, log)
    # the same call, one context, each call collected before the next is enqueued (what hm_call_chunks alone gives)
    sync_state = {}

    def step_sync():
        sync_state["rec"], sync_state["log"] = ctx.call_chunks(chunks, view=True, wait=False)

    step_sync()
    ms_sync = T.run(step_sync, args.steps, after=ctx.records_wait, streams=streams[:1]) / args.steps
    assert list(sync_state["log"]) == list(log)
    k_ms, launches = kernel_breakdown(ctx, step_sync)
    ctx.records_wait()
    # ---- end to end: the worker's call on the decoder's own buffers ----
    bam = os.path.join(tmpdir, "contig.bam")
    t0 = time.perf_counter()
    bamdec.write_batch_bam(bam, "chr1", len(d.ref), batch)
    t_write = time.perf_counter() - t0
    nb = bamdec.NativeBam(bam)
    t0 = time.perf_counter()
    dbatch, cq = nb.read_batch("chr1", 0, len(d.ref), copy=False, seq=False, compact=True)
    t_decode = time.perf_counter() - t0
    dchunks = dbatch.chunk_table(chunkloci(len(d.ref)))
    small = [getattr(dbatch, n) for n, _ in dbatch._FIELDS if n not in ("seq", "bq", "ops", "seq_off")]
    pinned = [cq.mask, cq.exc, cq.exc_off, dbatch.ops] + small
    ctx.pin_arrays(pinned)

    def step_e2e():
        state["rec_e"], state["log_e"] = ctx.call_batch_compact(dbatch, cq, dchunks, view=True)

    for _ in range(2):
        step_e2e()
    ms_e2e_one = T.run(step_e2e, args.steps, streams=streams[:1])
    assert list(state["log_e"]) == list(log), "the decoded batch gives other counters than the generated one"
    srt = lambda a: np.sort(a, order=["chunk", "tpos", "ref", "alt"]).tobytes()  # records come back in no particular order
    assert srt(state["rec_e"]) == srt(rec), "end-to-end records differ from the resident call's"
    # the same host buffers through the worker's two alternating contexts (himut_b200/caller.py:call_region): upload + submit
    # on one, then collect the other — the upload of a call overlaps the kernels and the record copy of the call before it
    e_state = {"k": 0, "pending": None}

    def step_e2e_alt():
        c = pair[e_state["k"] % 2]
        e_state["k"] += 1
        c.upload_compact(dbatch, cq, wait=False)  # enqueued before the previous upload is waited for, as the worker does
        if e_state["pending"] is not None:
            e_state["pending"].upload_wait()      # where the worker hands the previous group's buffers back to the decoder
        c.call_chunks_submit(dchunks)
        if e_state["pending"] is not None:
            e_state["rec"], e_state["log"] = e_state["pending"].call_chunks_collect(view=True)
        e_state["pending"] = c

    def drain_e2e():
        if e_state["pending"] is not None:
            e_state["pending"].upload_wait()
            e_state["rec"], e_state["log"] = e_state["pending"].call_chunks_collect(view=True)
            e_state["pending"] = None
        for c in pair:
            c.records_wait()

    for _ in range(4):
        step_e2e_alt()
    drain_e2e()
    ms_e2e = T.run(step_e2e_alt, args.steps, after=drain_e2e, streams=streams)
    assert list(e_state["log"]) == list(log) and srt(e_state["rec"]) == srt(rec), "pipelined end-to-end records differ from the resident call's"
    ctx_b.close()
    ctx.set_stream(T.stream.cuda_stream)
    h2d = int(cq.nbytes() + dbatch.ops.nbytes + sum(a.nbytes for a in small) + dchunks.nbytes)
    # the same call with one quality byte per base and the 2-bit bases (what round 1's workers uploaded)
    ctx.pin(batch)

    def step_plain():
        ctx.call_batch(batch, chunks, view=True)

    step_plain()
    ms_plain = T.run(step_plain, args.steps) / args.steps
    ctx.unpin(batch)
    ctx.unpin_arrays(pinned)
    nb.close()
    n_base, n_op, n_read = batch_counts(batch)
    alg = scan_alg_bytes(batch)
    peak, peak_src = measured_peak()
    scan_ms = k_ms.get("k_call_scan", float("nan"))
    dev_ms = float(sum(k_ms.values()))
    step_ms = ms_total / args.steps
    survey_bytes = 1.25 * n_base + 4.0 * n_op + 40.0 * n_read + 48.0 * rec.size
    out = {
        "value": aligned * args.steps / (ms_total * 1e-3), "ms_per_step": step_ms,
        "e2e": {"value": aligned * args.steps / (ms_e2e * 1e-3), "unit": "bases/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": int(rec.nbytes + 256), "ms_per_step": ms_e2e / args.steps,
                "call": "hm_upload_batch_compact_begin / hm_upload_wait + hm_call_chunks_submit / hm_call_chunks_collect on two alternating contexts: what "
                        "himut_b200/caller.py:call_region does from decode group to decode group (the upload of a call is enqueued before the previous "
                        "one is waited for and overlaps the kernels and the record copy of the call before it; every step uploads the "
                        "whole batch again and its records reach host memory inside the timed region); host buffers exactly as csrc/bamdec.c leaves them (no base stream, "
                        "qualities as modal bitmap + exceptions written by its record-parse pass), page-locked once before the loop; "
                        "records byte-identical to the resident call's",
                "one_context": {"value": aligned * args.steps / (ms_e2e_one * 1e-3), "ms_per_step": ms_e2e_one / args.steps,
                                "call": "hm_call_batch_compact on one context, each call finished before the next upload starts"},
                "decode_seconds_outside_timed_region": t_decode, "bam_write_seconds": t_write},
        "value_one_context": {"value": aligned / (ms_sync * 1e-3), "unit": "bases/s", "ms_per_step": ms_sync,
                              "call": "hm_call_chunks on one context, every call collected before the next is enqueued"},
        "value_call": "hm_call_chunks_submit / hm_call_chunks_collect on two contexts that alternate, the next call enqueued before the "
                      "previous is collected: how himut_b200/caller.py:call_region drives the device from decode group to decode group",
        "e2e_plain": {"value": aligned / (ms_plain * 1e-3), "unit": "bases/s", "h2d_bytes_per_step": int(batch.nbytes() + chunks.nbytes),
                      "ms_per_step": ms_plain, "call": "hm_call_batch: one quality byte per base + 2-bit bases (round 1's upload)"},
        "gpu_launches": int(launches * args.steps),
        "gpu_launches_per_step": int(launches),
        "library_launches_per_step": 0,
        "roofline": {"bound": "hbm", "kernel": "k_call_scan", "achieved": alg / (scan_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": alg / (scan_ms * 1e-3) / 1e9 / peak, "frac_of_nominal_8000_gbs": alg / (scan_ms * 1e-3) / 1e9 / 8000.0,
                     "traffic": ncu_traffic(alg),
                     "traffic_source": "profiles/traffic.json (ncu --set full, 64 Mb contig): ratio applied, not measured in this run",
                     "peak_source": peak_src, "alg_bytes_per_launch": alg, "kernel_ms": scan_ms,
                     "share_of_step_device_time": scan_ms / dev_ms if dev_ms else None,
                     # the whole step: SURVEY 8(d)'s bytes over the driver-comparable wall time of a step, and over its kernels alone
                     "frac_step": survey_bytes / (step_ms * 1e-3) / 1e9 / peak,
                     "frac_step_kernels_only": survey_bytes / (dev_ms * 1e-3) / 1e9 / peak if dev_ms else None,
                     "step_bytes_formula": "SURVEY 8(d): 1.25*N_base + 4*N_op + 40*N_read + 48*N_cand (the 0.25 B per base of the 2-bit "
                                           "stream is counted although `call` does not read it)",
                     "step_bytes": survey_bytes},
        "kernel_ms_per_step": k_ms, "kernel_ms_note": "CUDA events per kernel group, taken in 3 extra steps outside the timed loop",
        "aligned_bases_per_step": int(aligned), "site_records_per_step": int(rec.size),
        "records": "every record the reference emits (PASS + filtered sites) reaches host memory each step; germline restatements are "
                   "counted in the log on the device (HM_OPT_OMIT_RESTATEMENTS)",
        "log_counters": [int(v) for v in log],
    }
    return out, bam


def leg_phase(args, T, ctx, d):
    """BASELINE configs[3] on the same contig: `himut call --phase` with a phased germline table (phase sets of
    ~200 kb, chunks = their spans) and common-SNP + panel-of-normals sets, resident"""
    import cases
    from himut_b200 import gtmodel
    ph, spans, sets = cases.phase_case(d, 200_000)
    common, pon = cases.site_sets_from_synth(d, 3)
    p = gtmodel.make_params(**dict(gtmodel.DEFAULT_CALL_ARGS, phase=True))
    chunks = d.batch.chunk_table(spans, sets)
    ctx.set_params(p)
    ctx.set_site_sets(common, pon)
    ctx.set_phase_sets(ph)
    ctx.upload(d.batch.without_seq())
    state = {}

    def step():
        state["rec"], state["log"] = ctx.call_chunks(chunks, view=True, wait=False)

    for _ in range(2):
        step()
    n = args.steps
    ms = T.run(step, n, after=ctx.records_wait) / n
    k_ms, launches = kernel_breakdown(ctx, step)
    ctx.records_wait()
    rec, log = state["rec"], state["log"]
    out = {"value": d.aligned_bases / (ms * 1e-3), "unit": "bases/s", "ms_per_step": ms, "steps": n, "kernel_ms_per_step": k_ms,
           "phase_sets": len(spans), "hetsnps": int(ph["hpos"].size), "common_snps": int(common.size), "panel_of_normals": int(pon.size),
           "site_records_per_step": int(rec.size), "log_counters": [int(v) for v in log],
           "workload": "himut call --phase, phased germline table (phase sets of ~200 kb) + common-SNP + PoN sets, same 64 Mb contig"}
    # back to the plain configuration for the legs that follow
    ctx.set_params(gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS))
    ctx.set_site_sets()
    return out


def leg_normcounts(args, T, ctx, d, chunks):
    """the callable-base half of `himut normcounts` on the resident batch, uploaded as himut_b200/normcounts.py uploads
    it (qualities as modal bitmap + exceptions, expanded on the device); `plain_upload`: the same on a batch uploaded
    with one quality byte per base"""
    from himut_b200 import bamdec
    batch = d.batch
    n_norm = args.steps
    state = {}

    def step():
        state["r"] = ctx.normcounts_chunks(d.ref, chunks)

    def measure():
        ctx.normcounts_chunks(d.ref, chunks)
        ms = T.run(step, n_norm) / n_norm
        ctx.kernel_timing(True)
        step()
        nk = {k: v for k, v in ctx.last_kernel_times()}
        ctx.kernel_timing(False)
        return ms, nk

    ctx.upload(batch)
    ms_plain, nk_plain = measure()
    plain = state["r"]
    ctx.upload_compact(batch, bamdec.compact_bq(batch))
    ms, nk = measure()
    ccs_tri, ref_tri, nlog, nties = state["r"]
    same = all(np.array_equal(np.asarray(a), np.asarray(b)) for a, b in zip(plain[:3], state["r"][:3])) and plain[3] == nties
    n_base, n_op, n_read = batch_counts(batch)
    peak, _ = measured_peak()
    nbytes = 1.25 * n_base + 4.0 * n_op + 40.0 * n_read + 1.0 * len(d.ref)
    return {"value": d.aligned_bases / (ms * 1e-3), "unit": "bases/s", "ms_per_step": ms, "steps": n_norm, "kernel_ms_per_step": nk,
            "frac_step": nbytes / (ms * 1e-3) / 1e9 / peak,
            "step_bytes_formula": "SURVEY 8(d): 1.25*N_base + 4*N_op + 40*N_read + 1*N_refpos",
            "upload": "hm_upload_batch_compact (what himut_b200/normcounts.py does per decode group)",
            "plain_upload": {"value": d.aligned_bases / (ms_plain * 1e-3), "ms_per_step": ms_plain, "kernel_ms_per_step": nk_plain,
                             "frac_step": nbytes / (ms_plain * 1e-3) / 1e9 / peak, "same_result": bool(same)},
            "callable_bases": int(nlog[13]), "callable_positions": int(ref_tri.sum()), "alt_ties_flagged": int(nties),
            "positions_evaluated_exactly": ctx.last_norm_exact_sites(), "positions": int(len(d.ref)),
            "bound": "k_norm_prep: instruction issue (one pass over every read: bit vectors in reference coordinates); k_norm_bits: "
                     "latency; then the exact fp64 pass over the listed positions (sector gather), see DESIGN.md 4.1"}


def leg_bam_to_vcf(bam_path, contig_len, aligned_bases, tmp):
    """SURVEY 8(d) timing (ii): BAM on disk (page cache) -> VCF on disk through the worker mirror itself
    (himut_b200.caller.get_somatic_substitutions: native decode one group ahead, compact upload, device path, 12-tuples,
    natsort) and the mirror of the reference's writer (vcfio.dump_sbs).  Its own hm_ctx, like a worker process."""
    from himut_b200 import bamdec, caller, gtmodel, vcfio, worker
    a = gtmodel.DEFAULT_CALL_ARGS
    loci = [("chr1", s, e) for s, e in chunkloci(contig_len)]
    header = "##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tsynth"
    best = None
    for _ in range(3):
        lst, log = {}, {}
        t0 = time.perf_counter()
        caller.get_somatic_substitutions(
            "chr1", bam_path, None, None, loci, {}, {}, {}, a["min_qv"], a["min_mapq"], a["qlen_lower_limit"],
            a["qlen_upper_limit"], a["min_sequence_identity"], a["min_gq"], a["min_bq"], a["min_trim"], a["max_mismatch_count"],
            a["mismatch_window"], a["md_threshold"], a["min_ref_count"], a["min_alt_count"], a["min_hap_count"], 1e-6,
            a["germline_snv_prior"], 1e-4, False, True, False, lst, log)
        t1 = time.perf_counter()
        vcf = os.path.join(tmp, "out.vcf")
        vcfio.dump_sbs(vcf, header, ["chr1"], lst)
        t2 = time.perf_counter()
        if best is None or t2 - t0 < best[0]:
            best = (t2 - t0, t1 - t0, t2 - t1)
    return {"value": aligned_bases / best[0], "unit": "bases/s", "seconds": best[0], "worker_seconds": best[1],
            "writer_seconds": best[2], "rows": len(lst["chr1"]), "vcf_bytes": os.path.getsize(vcf), "contig_mb": contig_len // 1_000_000,
            "decode_threads": bamdec.default_threads(), "decode_group_mb": worker.GROUP_SPAN // 1_000_000,
            "bam_bytes": os.path.getsize(bam_path), "log": [int(v) for v in log["chr1"]],
            "note": "host bound: BGZF inflate + record parse on the host cores take most of it (decode of group k + 1 overlaps upload "
                    "and kernels of group k); non_human_sample = True (no common-SNP / PoN files)"}


# ------------------------------------------------------------------------------------------------ configs[2] (scaled)
def genome_contigs(genome_mb):
    scale = genome_mb / float(sum(HUMAN_MB))
    names = ["chr%d" % (i + 1) for i in range(22)] + ["chrX", "chrY"]
    return [(n, max(400_000, int(round(mb * scale * 5)) * 200_000)) for n, mb in zip(names, HUMAN_MB)]


def leg_genome(args, T, lib, torch, rank, world, local_rank, stream):
    """chunk runs of the scaled genome on this rank: resident and end-to-end timing, the 15 counters summed over ranks"""
    from concurrent.futures import ThreadPoolExecutor
    from himut_b200 import bamdec, genome, gtmodel, synth
    contigs = genome_contigs(args.genome_mb)
    loci = {c: genome.chunkloci(c, n) for c, n in contigs}
    runs = genome.plan_runs(loci, world)
    mine = [r for r in runs if r.rank == rank]
    order = [c for c, _ in contigs]
    need = sorted({r.chrom for r in mine}, key=order.index)
    length = dict(contigs)
    seed_of = {c: args.seed + 1009 * i for i, (c, _) in enumerate(contigs)}
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max(1, min(len(need), host_threads()))) as ex:
        data = dict(zip(need, ex.map(lambda c: synth.generate(length[c], seed=seed_of[c], copy=False), need)))
    t_gen = time.perf_counter() - t0
    params = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
    items, my_bases, streams = [], 0, []
    for r in mine:
        d = data[r.chrom]
        chunks_r = [(s, e) for _c, s, e in loci[r.chrom][r.lo:r.hi]]
        table_full = d.batch.chunk_table(chunks_r)
        lo, hi = int(table_full["read_lo"].min()), int(table_full["read_hi"].max())
        sub = slice_batch(d.batch, lo, hi)
        table = sub.chunk_table(chunks_r)
        cq = bamdec.compact_bq(sub)
        # aligned bases of the reads that START in the run: every read of the genome is counted once over all ranks
        a0 = -1 if r.lo == 0 else chunks_r[0][0]
        a1 = (1 << 31) - 1 if r.hi == len(loci[r.chrom]) else chunks_r[-1][1]
        per = aligned_per_read(sub)
        my_bases += int(per[(sub.tstart >= a0) & (sub.tstart < a1)].sum())
        # every run has two contexts of its own (each with its stream and the run's batch resident): they alternate from
        # step to step and the next step is enqueued before the previous one is collected, as himut_b200/caller.py drives
        # a worker's two contexts from decode group to decode group — so the device goes from run to run and from step
        # to step without waiting for the host, and collecting run k overlaps the kernels of the runs behind it.  The
        # timing events bracket all of it on the device (Timer.run: the streams wait for the opening event, the closing
        # event waits for the streams), barrier + synchronize on both sides.
        small = [getattr(sub, n) for n, _ in sub._FIELDS if n not in ("seq", "bq", "ops", "seq_off")]
        pinned = [cq.mask, cq.exc, cq.exc_off, sub.ops] + small
        pair = []
        for _k in range(2):
            ctx = lib.Context(local_rank)
            st = torch.cuda.Stream()
            ctx.set_stream(st.cuda_stream)
            streams.append(st)
            ctx.set_params(params)
            ctx.set_site_sets()
            ctx.omit_restatements(True)
            ctx.kernel_timing(False)
            if not pair:
                ctx.pin_arrays(pinned)
            ctx.upload_compact(sub, cq)
            pair.append(ctx)
        items.append(dict(ctx=pair[0], pair=pair, sub=sub, cq=cq, table=table, pinned=pinned, small=small, run=r))
    state = {"log": np.zeros(15, np.int64), "recs": 0, "k": 0, "pending": None}

    def collect(which):
        log, recs = np.zeros(15, np.int64), 0
        for it in items:
            rec, l = it["pair"][which].call_chunks_collect(view=True)
            log += l
            recs += rec.size
        state["log"], state["recs"] = log, recs

    def step():
        which = state["k"] % 2
        state["k"] += 1
        for it in items:
            it["pair"][which].call_chunks_submit(it["table"])
        if state["pending"] is not None:
            collect(state["pending"])
        state["pending"] = which

    def wait_all():
        if state["pending"] is not None:
            collect(state["pending"])
            state["pending"] = None
        for it in items:
            for c in it["pair"]:
                c.records_wait()

    for _ in range(2 * args.warmup + 4):
        step()
    wait_all()
    ms_res = T.run(step, args.steps, after=wait_all, streams=streams)

    def step_e2e():
        # host buffers -> device -> records, run by run; a run's kernels overlap the next run's upload (each run has its
        # own context and stream), every step ends with all records of the step in host memory
        prev = None
        for it in items:
            c = it["pair"][0]
            c.upload_compact(it["sub"], it["cq"], wait=False)  # begun before the previous run's upload is waited for
            if prev is not None:
                prev.upload_wait()
            c.call_chunks_submit(it["table"])
            if prev is not None:
                prev.call_chunks_collect(view=True)
            prev = c
        if prev is not None:
            prev.upload_wait()
            prev.call_chunks_collect(view=True)
        for it in items:
            it["pair"][0].records_wait()

    step_e2e()
    ms_e2e = T.run(step_e2e, args.steps, streams=streams)
    h2d = sum(int(it["cq"].nbytes() + it["sub"].ops.nbytes + sum(a.nbytes for a in it["small"]) + it["table"].nbytes) for it in items)
    d2h = int(state["recs"]) * 76 + 256 * len(items)
    for it in items:
        it["ctx"].kernel_timing(True)
    state["k"] = 0
    step()
    wait_all()
    launches = sum(it["ctx"].last_timing()[1] for it in items)
    for it in items:
        assert it["ctx"].last_call_path() == 2
        it["ctx"].unpin_arrays(it["pinned"])
        for c in it["pair"]:
            c.close()
    dev = torch.device("cuda", local_rank)
    t = torch.tensor([ms_res, ms_e2e], device=dev, dtype=torch.float64)
    s = torch.tensor([float(my_bases), float(state["recs"]), float(h2d), float(d2h), float(launches), float(len(items))], device=dev,
                     dtype=torch.float64)
    mx = torch.tensor([float(my_bases)], device=dev, dtype=torch.float64)
    logt = torch.tensor(state["log"], device=dev)
    per_rank = [[ms_res / args.steps, ms_e2e / args.steps, float(my_bases), float(state["recs"]) * 76.0]]
    if world > 1:
        mine_t = torch.tensor(per_rank[0], device=dev, dtype=torch.float64)
        allt = [torch.zeros_like(mine_t) for _ in range(world)]
        T.dist.all_gather(allt, mine_t)
        per_rank = [[float(v) for v in x.tolist()] for x in allt]
        T.dist.all_reduce(t, op=T.dist.ReduceOp.MAX)
        T.dist.all_reduce(s, op=T.dist.ReduceOp.SUM)
        T.dist.all_reduce(mx, op=T.dist.ReduceOp.MAX)
        T.dist.all_reduce(logt, op=T.dist.ReduceOp.SUM)  # the only cross-GPU step of the path: 15 counters
    bases = float(s[0])
    return {
        "value": bases * args.steps / (float(t[0]) * 1e-3), "ms_per_step": float(t[0]) / args.steps,
        "e2e": {"value": bases * args.steps / (float(t[1]) * 1e-3), "unit": "bases/s", "ms_per_step": float(t[1]) / args.steps,
                "h2d_bytes_per_step": int(s[2]), "d2h_bytes_per_step": int(s[3]),
                "call": "hm_upload_batch_compact_begin / hm_upload_wait + hm_call_chunks_submit / collect per chunk run (a run's upload is begun before the previous run's is waited for, a run's kernels overlap the next run's "
                        "upload), host buffers in the decoder's layout (no base stream, qualities as modal "
                        "bitmap + exceptions — here built by hm_bq_compact_build from the generated batch, the same bytes the decoder's "
                        "parse pass writes: tests/test_bamdec.py), page-locked before the loop"},
        "aligned_bases_per_step": int(bases), "site_records_per_step": int(s[1]), "runs": len(runs), "runs_this_rank": len(items),
        "split_contigs": sum(1 for c in loci if sum(1 for r in runs if r.chrom == c) > 1),
        "imbalance": {"max_over_mean_bases_per_rank": float(mx[0]) / (bases / world) if bases else None,
                      "planned_max_over_mean_weight": genome.imbalance(runs, world)},
        "gpu_launches_per_step": int(s[4]), "contexts": int(s[5]), "generate_seconds_this_rank": t_gen,
        "per_rank": {"ms_per_step": [round(x[0], 4) for x in per_rank], "e2e_ms_per_step": [round(x[1], 4) for x in per_rank],
                     "aligned_bases": [int(x[2]) for x in per_rank], "record_bytes_d2h_per_step": [int(x[3]) for x in per_rank],
                     "record_d2h_gbs_if_it_were_the_only_limit": [round(x[3] / (x[0] * 1e-3) / 1e9, 2) if x[0] else None for x in per_rank]},
        "log_counters_sum": [int(v) for v in logt.tolist()],
        "log_note": "summed over runs: a candidate on the one position two runs of a split contig share is counted by both (the "
                    "product path, himut_b200/genome.py, replays som_seen over it at the merge; tests/test_zz_gpu_genome.py)",
    }


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--contig-mb", type=int, default=64)
    ap.add_argument("--genome-mb", type=int, default=776, help="size of the scaled configs[2] genome (3.1 Gb / 4)")
    ap.add_argument("--seed", type=int, default=20260101)
    ap.add_argument("--cpu-chunks", type=int, default=25)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-normcounts", action="store_true")
    ap.add_argument("--no-bam-leg", action="store_true")
    ap.add_argument("--no-genome", action="store_true")
    ap.add_argument("--no-phase", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the records and log counters of the headline call's last step as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (world > 1 or args.impl != "ours"):
        ap.error("--dump-outputs writes the one-GPU headline call's outputs: N = 1 and --impl ours only")

    import __graft_entry__ as g
    if args.impl == "reference":
        g.build(load=False)  # the CPU arm: nothing of the product is loaded
        return run_reference(args, rank, world)
    g.build()

    import torch
    import torch.distributed as dist
    from himut_b200 import lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    bind_to_gpu_numa_node(local_rank)
    saved_stdout = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        # stdout carries the one JSON line only: NCCL prints its version banner there when the first communicator comes up
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.current_stream()
    T = Timer(torch, dist, world, stream)
    sampler = ClockSampler(local_rank)
    tmpdir = tempfile.mkdtemp(prefix="himut_b200_bench_")
    out = None
    try:
        if world == 1:
            contig_len = args.contig_mb * 1_000_000
            d, params, chunks = make_workload(contig_len, args.seed)
            ctx = lib.Context(local_rank)
            ctx.set_stream(stream.cuda_stream)
            sampler.start()
            res, bam = leg_contig(args, T, ctx, d, params, chunks, tmpdir)
            clocks = sampler.stop()  # sampled over the resident and the end-to-end loops of the headline
            out = {"metric": METRIC, "value": res.pop("value"), "unit": "bases/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
                   "ms_per_step": res.pop("ms_per_step"), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                   "dtype": "u8/f64", "data": "synthetic", "config": workload_config(args, 1), "clocks": clocks}
            out.update(res)
            if not args.no_phase:
                try:
                    out["phase"] = leg_phase(args, T, ctx, d)
                except Exception as ex:
                    out["phase"] = {"error": repr(ex)}
            if not args.no_normcounts:
                try:
                    out["normcounts"] = leg_normcounts(args, T, ctx, d, chunks)
                except Exception as ex:  # a side measurement: never costs the line
                    out["normcounts"] = {"error": repr(ex)}
            ctx.close()
            if not args.no_bam_leg:
                try:
                    out["bam_to_vcf"] = leg_bam_to_vcf(bam, contig_len, d.aligned_bases, tmpdir)
                except Exception as ex:  # a side measurement: never costs the line
                    out["bam_to_vcf"] = {"error": repr(ex)}
            if not args.no_cpu_baseline:
                threads = host_threads()
                n = max(1, min(len(chunks) // threads, args.cpu_chunks))
                v1, bases1, dt1, _ = cpu_baseline(d, params, chunks, n, 1)
                v, bases, dt, used = cpu_baseline(d, params, chunks, n, threads)
                out["cpu_baseline"] = {"value": v, "unit": "bases/s", "cores": used, "kind": "port",
                                       "sample": "%d threads x %d consecutive chunks of %d (%d aligned bases, %.1f s) of the same contig"
                                                 % (used, n, len(chunks), bases, dt),
                                       "one_core": {"value": v1, "bases": bases1, "seconds": dt1}, "note": PY_REF_NOTE}
            del d
            if not args.no_genome:
                try:
                    out["genome"] = leg_genome(args, T, lib, torch, rank, world, local_rank, stream)
                    out["genome"]["workload"] = workload_config(args, 2)["workload"].replace("sharded over 2 GPUs", "planned for N GPUs (here: all on this one)")
                    out["genome"]["note"] = ("strong-scaling base of the N > 1 lines (whose headline is this workload): efficiency(N) = "
                                             "value(N) / (N x this value)")
                except Exception as ex:
                    out["genome"] = {"error": repr(ex)}
        else:
            if rank == 0:
                sampler.start()  # one sampler for the job: eight concurrent NVML pollers slow every rank's driver calls down
            res = leg_genome(args, T, lib, torch, rank, world, local_rank, stream)
            clocks = sampler.stop() if rank == 0 else None
            if rank == 0:
                out = {"metric": METRIC, "value": res.pop("value"), "unit": "bases/s", "n_gpus": world, "steps": args.steps,
                       "warmup": args.warmup, "ms_per_step": res.pop("ms_per_step"), "higher_is_better": True, "scaling": "strong",
                       "vs_baseline": None, "dtype": "u8/f64", "data": "synthetic", "config": workload_config(args, world), "clocks": clocks,
                       "gpu_launches": int(res["gpu_launches_per_step"] * args.steps)}
                out.update(res)
                out["scaling_note"] = ("strong scaling: the same %d Mb genome for every N > 1; its one-GPU base is the `genome` object of "
                                       "the N = 1 line (whose headline is BASELINE configs[1], a different workload)" % args.genome_mb)
        if saved_stdout is not None:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
            saved_stdout = None
        if rank == 0 and out is not None:
            print(json.dumps(out))
            sys.stdout.flush()
    finally:
        import shutil
        shutil.rmtree(tmpdir, ignore_errors=True)
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
