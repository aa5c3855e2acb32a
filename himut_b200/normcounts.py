"""GPU worker of `himut normcounts` (callable-base half): drop-in for
himut.normcounts.get_callable_tricounts (src/himut/normcounts.py:206-420).

Fills chrom2ccs_callable_tri2count[chrom], chrom2ref_callable_tri2count[chrom] (keys in
mutlib.tri_lst order; contexts containing N are tallied under "NNN", which the reference's
consumers never read, mutlib.py:2384-2393) and chrom2norm_log[chrom] (14 counters).
"""
import numpy as np

from . import abi, gtmodel, vcfio, worker

# mutlib.tri_lst (src/himut/mutlib.py:17-50)
TRI_LST = [a + c + b for a in "ACGT" for c in "CT" for b in "ACGT"]

# compressed BAM bytes per decode group from which normcounts_region(decode="auto") decodes on the device.  The worker
# is faster on the device decoder at every size measured (profiles/decode_trace_norm_r04.json): 22 ms vs 29 ms on the
# 1 Mb BAM (15.6 MB, one group), although the decode alone is slower there (15.7 ms vs 8.8 ms), because the host path
# still uploads the bases and the compact qualities and expands them; smaller groups are not measured and stay on the
# host decoder.
DEVICE_DECODE_MIN_BYTES = 14 << 20


def normcounts_region(ctx, bam_file, chrom, refseq, chunkloci_lst, chunk_sets, decode="auto"):
    """the device path of normcounts over a contig's chunk list, decode group by decode group.
    decode: "device" inflates and parses each group on the GPU from the compressed file with the 2-bit base stream
    (Context.decode_region(..., seq=True)); "host" decodes with the native host decoder one group ahead of the device;
    "auto" takes the device decoder when the groups average at least DEVICE_DECODE_MIN_BYTES of compressed BAM.  Either
    needs a context with the device decoder and a BAM with a BAI; without them the host decoder runs.
    -> (ccs_tri[33], ref_tri[33], log[14], n_alt_tie, distinct query names that passed the read gates); log[0] is
    that count"""
    src = worker.RegionSource(bam_file)
    tally = worker.QnameTally()
    ccs = np.zeros(abi.TRI_BINS, np.int64)
    ref = np.zeros(abi.TRI_BINS, np.int64)
    log = np.zeros(abi.NORM_LOG_LEN, np.int64)
    ties = 0
    groups = worker.group_chunks(chunkloci_lst)
    lo, hi = (min(s for _, s, _e in chunkloci_lst), max(e for _, _s, e in chunkloci_lst)) if chunkloci_lst else (None, None)

    def add(table):
        nonlocal ties
        c, r, l, t = ctx.normcounts_chunks(refseq, table)
        tally.add(ctx.qname_seen())
        ccs[:] += c; ref[:] += r; log[:] += l
        ties += t

    try:
        decode = worker.choose_decode(decode, ctx, src.reader, chrom, lo, hi, len(groups), DEVICE_DECODE_MIN_BYTES)
        if decode == "device":
            for idx in groups:
                loci = [chunkloci_lst[i] for i in idx]
                region = ctx.decode_region(src.reader, chrom, min(s for _, s, _e in loci), max(e for _, _s, e in loci), seq=True)
                if region.n_reads == 0:
                    continue
                add(region.chunk_table([(s, e) for _, s, e in loci], None if chunk_sets is None else [chunk_sets[i] for i in idx]))
        else:
            pins = worker.PinCache(ctx, enabled=len(groups) > 1)
            try:
                # qualities in the decoder's compact form, bases as a stream (the tile kernel reads them), decode one group ahead
                for _idx, batch, cq, table, release in worker.pipelined_groups(src, chrom, chunkloci_lst, groups, chunk_sets, seq=True):
                    if batch.n_reads == 0:
                        release()
                        continue
                    pins.pin([cq.mask, cq.exc, batch.ops, batch.seq])
                    ctx.upload_compact(batch, cq)
                    release()
                    add(table)
            finally:
                pins.close()
    finally:
        src.close()
    log[0] = tally.count()
    return ccs, ref, log, ties, int(log[0])


def get_callable_tricounts(
    chrom, seq, bam_file, common_snps, panel_of_normals, chunkloci_lst, phase_set2hbit_lst, phase_set2hpos_lst,
    phase_set2hetsnp_lst, min_qv, min_mapq, min_trim, qlen_lower_limit, qlen_upper_limit, min_sequence_identity,
    min_gq, min_bq, mismatch_window, max_mismatch_count, min_ref_count, min_alt_count, min_hap_count, md_threshold,
    somatic_snv_prior, germline_snv_prior, germline_indel_prior, phase, non_human_sample,
    chrom2ccs_callable_tri2count, chrom2ref_callable_tri2count, chrom2norm_log,
):
    ctx = worker.context()
    params = gtmodel.make_params(
        min_qv=min_qv, min_mapq=min_mapq, qlen_lower_limit=qlen_lower_limit, qlen_upper_limit=qlen_upper_limit,
        min_sequence_identity=min_sequence_identity, min_gq=min_gq, min_bq=min_bq, min_trim=min_trim,
        max_mismatch_count=max_mismatch_count, mismatch_window=mismatch_window, md_threshold=md_threshold,
        min_ref_count=min_ref_count, min_alt_count=min_alt_count, min_hap_count=min_hap_count,
        germline_snv_prior=germline_snv_prior, phase=phase, non_human_sample=non_human_sample)
    ctx.set_params(params)
    # normcounts loads both sets whenever a file is given (normcounts.py:248-289)
    ctx.set_site_sets(vcfio.load_common_snps(chrom, common_snps), vcfio.load_pon(chrom, panel_of_normals))
    chunk_sets = None
    if phase:
        table, chunk_sets = vcfio.phase_tables(chunkloci_lst, phase_set2hbit_lst, phase_set2hpos_lst, phase_set2hetsnp_lst)
        ctx.set_phase_sets(table)
    refseq = seq.encode() if isinstance(seq, str) else bytes(seq)
    ccs, ref, log, ties, _ = normcounts_region(ctx, bam_file, chrom, refseq, chunkloci_lst, chunk_sets)
    ccs_d = {tri: int(ccs[i]) for i, tri in enumerate(TRI_LST)}
    ref_d = {tri: int(ref[i]) for i, tri in enumerate(TRI_LST)}
    if ccs[32] or ref[32]:
        ccs_d["NNN"], ref_d["NNN"] = int(ccs[32]), int(ref[32])
    chrom2ccs_callable_tri2count[chrom] = ccs_d
    chrom2ref_callable_tri2count[chrom] = ref_d
    chrom2norm_log[chrom] = [int(v) for v in log]
    return ties
