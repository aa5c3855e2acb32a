"""Shared machinery of the two worker mirrors: one lazily created context per process, the
region -> packed batch step, and chunk grouping so a contig never has to fit in one batch."""
import os

import numpy as np

from . import abi, bamdec, lib

_CTX = None
_CTX_PID = None

# upper bound of reference span decoded into one batch (30x, compact qualities -> ~0.12 GB per 16 Mb); a contig longer
# than this is fed in several groups, decoded one ahead of the device (pipelined_groups)
GROUP_SPAN = int(os.environ.get("HIMUT_B200_GROUP_SPAN", 16_000_000))


def context():
    """the process's hm_ctx, created on first use *inside* the worker process (fork safe).
    Device: HIMUT_B200_DEVICE, else LOCAL_RANK, else worker index modulo visible GPUs."""
    global _CTX, _CTX_PID
    if _CTX is None or _CTX_PID != os.getpid():
        dev = os.environ.get("HIMUT_B200_DEVICE", os.environ.get("LOCAL_RANK"))
        if dev is None:
            import multiprocessing as mp
            ident = mp.current_process()._identity
            dev = (ident[0] - 1) if ident else 0
            n = int(os.environ.get("HIMUT_B200_NUM_DEVICES", "0")) or _device_count()
            dev = dev % max(n, 1)
        _CTX = lib.Context(int(dev))
        _CTX_PID = os.getpid()
        if os.environ.get("HIMUT_B200_VERBOSE"):
            import sys
            print("himut_b200: worker %d uses CUDA device %d" % (os.getpid(), int(dev)), file=sys.stderr)
    return _CTX


_CTX2 = None


def second_context():
    """a second hm_ctx on the process's device: the worker mirrors alternate between the two from decode group to
    decode group, so the upload of group k + 1 overlaps the kernels of group k (each context has its own stream)"""
    global _CTX2
    first = context()
    if _CTX2 is None or _CTX2[0] != os.getpid() or _CTX2[2] is not first:
        _CTX2 = (os.getpid(), lib.Context(first.device), first)
    return _CTX2[1]


def _device_count():
    """visible CUDA devices, asked of the library itself (cudaGetDeviceCount): no torch import in a pool worker"""
    return max(1, lib.device_count())


def group_chunks(chunkloci_lst, span=None):
    """consecutive chunks grouped so each group's decoded window stays under `span` bases"""
    span = span or GROUP_SPAN
    groups, cur, lo, hi = [], [], None, None
    for i, (_c, s, e) in enumerate(chunkloci_lst):
        nlo = s if lo is None else min(lo, s)
        nhi = e if hi is None else max(hi, e)
        if cur and nhi - nlo > span:
            groups.append(cur)
            cur, nlo, nhi = [], s, e
        cur.append(i)
        lo, hi = nlo, nhi
    if cur:
        groups.append(cur)
    return groups


def choose_decode(decode, ctx, reader, chrom, lo, hi, n_groups, min_bytes):
    """which decoder reads [lo, hi) of chrom in n_groups groups: "device" (Context.decode_region) or "host" (the
    native host decoder).  "device" needs a context with the device decoder and a BAM with a BAI, else the host
    decoder runs; "auto" also needs the groups to average at least min_bytes of compressed BAM (below that the host
    decoder's threads finish first).  lo None: nothing to decode."""
    if decode not in ("auto", "host", "device"):
        raise ValueError("decode must be 'auto', 'host' or 'device'")
    if decode != "host" and not (hasattr(ctx, "decode_region") and reader.has_index):
        return "host"
    if decode == "auto":
        if lo is None:
            return "host"
        return "device" if reader.plan(chrom, lo, hi).comp_bytes >= min_bytes * n_groups else "host"
    return decode


class RegionSource:
    """decodes the records a group of chunks fetches into one packed batch"""

    def __init__(self, bam_file):
        # native decoder (csrc/bamdec.c): threaded BGZF inflate, record parse and cs -> ops in C;
        # query-name ids are interned per handle, so they stay global across groups
        # (num_ccs counts distinct names per contig)
        self.reader = bamdec.NativeBam(bam_file)

    def batch(self, chrom, chunkloci, phase_sets=None, seq=True, compact=False, buffer_set=0, pad=0):
        """seq=False: without the 2-bit base stream (`call`, phase edges: ReadBatch.without_seq says why).
        compact=True: -> (batch, abi.BqCompact, table), the qualities as the decoder's parse pass writes them for the
        upload (bitmap + exceptions).  pad: decode that many positions past the last chunk end (`call --phase`
        re-fetches [tpos, tpos + 1) at a site, which reaches one position past a chunk that ends at tpos)."""
        lo = min(s for _, s, _e in chunkloci)
        hi = max(e for _, _s, e in chunkloci) + pad
        got = self.reader.read_batch(chrom, lo, hi, copy=False, seq=seq, compact=compact, buffer_set=buffer_set)
        batch, cq = got if compact else (got, None)
        table = batch.chunk_table([(s, e) for _, s, e in chunkloci], phase_sets)
        return (batch, cq, table) if compact else (batch, table)

    def close(self):
        self.reader.close()


def pipelined_groups(src, chrom, chunkloci_lst, groups, chunk_sets, seq, pad=0):
    """the groups of a contig, decoded one ahead of the consumer on a thread of their own (the decoder's C calls drop
    the GIL): decode(k + 1) runs while group k is uploaded and called.  The decoder's two buffer sets alternate; the
    consumer hands a set back with release() as soon as its upload has returned (hm_upload_batch* copies everything).
    Yields (idx, batch, cq, table, release)."""
    import queue
    import threading
    if len(groups) == 1:  # nothing to overlap
        idx = groups[0]
        b, cq, t = src.batch(chrom, [chunkloci_lst[i] for i in idx], None if chunk_sets is None else [chunk_sets[i] for i in idx],
                             seq=seq, compact=True, pad=pad)
        yield idx, b, cq, t, (lambda: None)
        return
    free, ready = queue.Queue(), queue.Queue()
    free.put(0); free.put(1)
    stop = threading.Event()

    def work():
        try:
            for idx in groups:
                s = free.get()
                if stop.is_set():
                    return
                loci = [chunkloci_lst[i] for i in idx]
                b, cq, t = src.batch(chrom, loci, None if chunk_sets is None else [chunk_sets[i] for i in idx],
                                     seq=seq, compact=True, buffer_set=s, pad=pad)
                ready.put((idx, b, cq, t, s))
            ready.put(None)
        except BaseException as ex:  # delivered to the consumer
            ready.put(ex)

    th = threading.Thread(target=work, name="himut-b200-decode", daemon=True)
    th.start()
    try:
        while True:
            item = ready.get()
            if item is None:
                break
            if isinstance(item, BaseException):
                raise item
            idx, b, cq, t, s = item
            yield idx, b, cq, t, (lambda s=s: free.put(s))
    finally:
        stop.set()
        free.put(0)  # unblock a decoder waiting for a set
        th.join()


class PinCache:
    """page-locks the decoder's big output buffers once per (address, size): they are reused from group to group, so
    the H2D copies of every group but the first run at PCIe speed.  Opt-in (HIMUT_B200_PIN_DECODE=1): on the B200 boxes
    measured (VMs), cudaHostRegister of a contig's two buffer sets (0.45 GB) takes 0.6 - 4 s, where the pageable copies it
    saves take under 0.1 s per 64 Mb contig and the decode itself 0.5 s (tools/worker_trace.py)."""

    def __init__(self, ctx, enabled):
        self.ctx, self.held = ctx, {}
        self.enabled = enabled and os.environ.get("HIMUT_B200_PIN_DECODE", "0") not in ("", "0")

    def pin(self, arrays):
        if not self.enabled:
            return
        for a in arrays:
            if a is None or a.nbytes < (1 << 22):
                continue
            key = a.ctypes.data
            old = self.held.get(key)
            if old is not None and old.nbytes >= a.nbytes:
                continue
            if old is not None:
                self.ctx.unpin_arrays([old])
            self.ctx.pin_arrays([a])
            self.held[key] = a

    def close(self):
        if self.held:
            self.ctx.unpin_arrays(list(self.held.values()))
            self.held = {}


class Laps:
    """wall-clock laps of a worker's host loop, reported to stderr when HIMUT_B200_WORKER_TIMING is set (diagnostics)"""

    def __init__(self, title):
        self.on = bool(os.environ.get("HIMUT_B200_WORKER_TIMING"))
        self.title, self.acc = title, {}
        if self.on:
            import time
            self.clock = time.perf_counter
            self.t = self.t0 = self.clock()

    def __call__(self, name):
        if self.on:
            now = self.clock()
            self.acc[name] = self.acc.get(name, 0.0) + now - self.t
            self.t = now

    def report(self):
        if self.on:
            import sys
            print("[%s] %.3f s: %s" % (self.title, self.clock() - self.t0, ", ".join("%s %.3f" % kv for kv in self.acc.items())),
                  file=sys.stderr)


class QnameTally:
    """distinct query names that passed the read gates, across groups (m.num_ccs)"""

    def __init__(self):
        self.seen = np.zeros(0, np.uint8)

    def add(self, flags):
        if flags.size > self.seen.size:
            self.seen = np.concatenate([self.seen, np.zeros(flags.size - self.seen.size, np.uint8)])
        self.seen[: flags.size] |= flags

    def count(self):
        return int(np.count_nonzero(self.seen))
