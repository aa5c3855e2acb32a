"""GPU worker of `himut phase`'s edge counting: drop-in for himut.phaselib.get_edges
(src/himut/phaselib.py:16-67, SURVEY.md §8f row 4).

Same arguments, same return value: (natsorted list of (i, j) edges, {(i, j): np.array of the four
cis / trans counts}).  The BAM is decoded window by window, on the device or the host (edge_table; a read that two
windows share is counted with the window it starts in), the pair tables are accumulated on the device in a band
(hm_phase_edges_*), and only non-empty tables become dictionary entries — the reference creates an
entry when it first increments it.  The binomial tests and the BFS over the graph stay the
reference's own code (phaselib.py:70-195).
"""
from collections import defaultdict

import numpy as np

from . import caller, natsort_compat, worker

BASE2CODE = {"A": 0, "T": 1, "G": 2, "C": 3}


def edge_table(ctx, bam_file, chrom, hpos, href, min_bq, min_mapq, decode="auto"):
    """the pair tables of the hetSNPs (hpos, href) over the whole contig, decoded window by window (worker.GROUP_SPAN)
    -> uint32[n_hetsnp, band, 4] (Context.phase_edges_end).
    decode: "device" decodes each window on the GPU from the compressed file (Context.decode_region, no base stream);
    "host" with the native host decoder; "auto" takes the device decoder when the windows average at least
    caller.DEVICE_DECODE_MIN_BYTES of compressed BAM (the same no-seq decode that threshold was measured on).  Either
    needs a context with the device decoder and a BAM with a BAI; without them the host decoder runs."""
    src = worker.RegionSource(bam_file)
    try:
        length = src.reader.lengths[src.reader.references.index(chrom)]
        n_windows = -(-length // worker.GROUP_SPAN)
        decode = worker.choose_decode(decode, ctx, src.reader, chrom, 0 if length else None, length, n_windows,
                                      caller.DEVICE_DECODE_MIN_BYTES)
        band = 64
        while True:
            ctx.phase_edges_begin(hpos, href, band)
            need, lo = 0, 0
            while lo < length and not need:
                hi = min(length, lo + worker.GROUP_SPAN)
                if decode == "device":
                    n_reads = ctx.decode_region(src.reader, chrom, lo, hi).n_reads
                else:
                    batch, _ = src.batch(chrom, [(chrom, lo, hi)], seq=False)  # a cs match at a hetSNP carries its reference allele
                    n_reads = batch.n_reads
                    if n_reads:
                        ctx.upload(batch)
                if n_reads:
                    need = ctx.phase_edges_add(min_bq, min_mapq, lo if lo else -2**31)
                lo = hi
            if not need:
                break
            band = max(need, band * 2)  # a read paired hetSNPs further apart than the band: start over, wider
        return ctx.phase_edges_end()
    finally:
        src.close()


def get_edges(chrom, bam_file, min_bq, min_mapq, hpos_lst, hetsnp_lst, hetsnp2hidx):
    try:
        from natsort import natsorted
    except ImportError:  # pragma: no cover - natsort is a dependency of the reference
        natsorted = natsort_compat.natsorted
    edge2counts = defaultdict(lambda: np.zeros(4))
    n = len(hpos_lst)
    if n >= 2:
        hpos = np.asarray(hpos_lst, np.int32)
        href = np.array([BASE2CODE.get(h[1], 4) for h in hetsnp_lst], np.uint8)
        hidx = np.array([hetsnp2hidx[h] for h in hetsnp_lst], np.int64)
        table = edge_table(worker.context(), bam_file, chrom, hpos, href, min_bq, min_mapq)
        a_idx, d_idx = np.nonzero(table.any(axis=2))
        for a, d in zip(a_idx.tolist(), d_idx.tolist()):
            edge2counts[(int(hidx[a]), int(hidx[a + d + 1]))] += table[a, d].astype(np.float64)
    edge_lst = natsorted(list(edge2counts.keys()))
    return edge_lst, edge2counts
