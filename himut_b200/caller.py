"""GPU worker of `himut call`: drop-in for himut.caller.get_somatic_substitutions.

Same positional signature, same contract as the reference worker (src/himut/caller.py:208-642):
it fills chrom2tsbs_lst[chrom] with the natsorted 12-tuples and chrom2tsbs_log[chrom] with the
15 counters.  Install with himut_b200.patch.install() (see INTEGRATION.md).
"""
import numpy as np

from . import abi, gtmodel, records, vcfio, worker

_RESTATES = (abi.ST_GERM_HET, abi.ST_GERM_HETALT, abi.ST_GERM_HOMALT, abi.ST_GERM_HOMREF)

# compressed BAM bytes per decode group from which call_region(decode="auto") decodes on the device: below it the host
# decoder's threads finish a group first (tools/decode_trace.py, profiles/decode_trace_r03.json)
DEVICE_DECODE_MIN_BYTES = 48 << 20


def _log_from_records(rec, num_ccs):
    """chrom2tsbs_log vector (caller.py:625-641) from record statuses"""
    h = np.bincount(rec["status"], minlength=16).astype(np.int64)
    log = np.zeros(abi.CALL_LOG_LEN, np.int64)
    log[0] = num_ccs
    log[1] = rec.size
    log[2], log[3], log[4] = h[abi.ST_GERM_HET], h[abi.ST_GERM_HETALT], h[abi.ST_GERM_HOMALT]
    log[5] = h[abi.ST_HET_SITE] + h[abi.ST_HETALT_SITE] + h[abi.ST_HOMALT_SITE]
    log[7] = h[abi.ST_INDEL_SITE]
    log[8], log[9], log[10], log[11] = h[abi.ST_LOW_GQ], h[abi.ST_LOW_BQ], h[abi.ST_PON], h[abi.ST_COMSNP]
    log[12], log[13] = h[abi.ST_HIGH_DEPTH], h[abi.ST_LOW_DEPTH]
    log[14] = h[abi.ST_PASS] + h[abi.ST_UNPHASED]
    log[6] = log[8:15].sum()
    return log


def configure(ctx, chrom, common_snps, panel_of_normals, chunkloci_lst, phase_set2hbit_lst, phase_set2hpos_lst, phase_set2hetsnp_lst,
              min_qv, min_mapq, qlen_lower_limit, qlen_upper_limit, min_sequence_identity, min_gq, min_bq, min_trim,
              max_mismatch_count, mismatch_window_size, md_threshold, min_ref_count, min_alt_count, min_hap_count,
              germline_snv_prior, phase, non_human_sample, create_panel_of_normals):
    """worker arguments -> context state (parameters, site sets, phase table); returns the phase-set index per chunk"""
    params = gtmodel.make_params(
        min_qv=min_qv, min_mapq=min_mapq, qlen_lower_limit=qlen_lower_limit, qlen_upper_limit=qlen_upper_limit,
        min_sequence_identity=min_sequence_identity, min_gq=min_gq, min_bq=min_bq, min_trim=min_trim,
        max_mismatch_count=max_mismatch_count, mismatch_window=mismatch_window_size, md_threshold=md_threshold,
        min_ref_count=min_ref_count, min_alt_count=min_alt_count, min_hap_count=min_hap_count,
        germline_snv_prior=germline_snv_prior, phase=phase, non_human_sample=non_human_sample,
        create_panel_of_normals=create_panel_of_normals)
    ctx.set_params(params)
    # the reference only loads the sets when neither flag is given (caller.py:248-289)
    if non_human_sample or create_panel_of_normals:
        ctx.set_site_sets()
    else:
        ctx.set_site_sets(vcfio.load_common_snps(chrom, common_snps), vcfio.load_pon(chrom, panel_of_normals))
    chunk_sets = None
    if phase:
        table, chunk_sets = vcfio.phase_tables(chunkloci_lst, phase_set2hbit_lst, phase_set2hpos_lst, phase_set2hetsnp_lst)
        ctx.set_phase_sets(table)
    return chunk_sets


def carry_som_seen(parts, later_starts):
    """som_seen across consecutive pieces of one contig's chunk list (groups of a worker, runs of a sharded job), as it
    carries across chunks (caller.py:243,347; bamlib.py:77): a candidate whose position an earlier piece claimed is
    dropped, a piece claims the positions of its records that are not germline restatements.
    parts: record arrays in chunk order; later_starts[i]: the smallest chunk start after piece i (None: nothing
    follows) — only positions at or past it can matter later.  Returns the filtered arrays."""
    som_seen, out = set(), []
    for rec, later in zip(parts, later_starts):
        if som_seen and rec.size:
            rec = rec[~np.isin(rec["tpos"], np.fromiter(som_seen, np.int32, len(som_seen)))]
        if later is not None and rec.size:
            claim = rec[(~np.isin(rec["status"], _RESTATES)) & (rec["tpos"] >= later)]
            som_seen.update(int(t) for t in claim["tpos"])
        out.append(rec)
    return out


def call_region(ctx, bam_file, chrom, chunkloci_lst, chunk_sets, phase, want_names=False, ctx2=None, decode="auto", refseq=None):
    """the device path over a contig's chunk list (or a run of it), pipelined: group k + 1 is decoded on a thread of its
    own while group k is uploaded; with a second context (configured like the first) the two alternate from group to
    group, so upload(k + 1) also overlaps kernels(k) and the record copy of k - 1:
        decode(k + 1) || H2D(k + 1) || kernels(k) || D2H(k - 1).
    decode: "device" inflates and parses each group on the GPU from the compressed file (Context.decode_region): the
    context that calls a group decodes it, and with two contexts the decode of group k + 1 runs while the kernels of
    group k do.  It needs a context with the device decoder and a BAM with a BAI; without either the host decoder runs.
    "host" is the pipeline above (the native host decoder).  "auto" takes the device decoder when it can run and the
    groups average at least DEVICE_DECODE_MIN_BYTES of compressed BAM (below that the host decoder is faster).
    refseq: the sequence of `chrom`, for records with neither cs:Z nor MD:Z, which whichever decoder runs then decodes
    from CIGAR + reference (every context that decodes gets it); None: such records are rejected.
    -> (records incl. germline restatements, number of distinct query names that passed the read gates,
        names blob (want_names) or None)"""
    if decode not in ("auto", "host", "device"):
        raise ValueError("decode must be 'auto', 'host' or 'device'")
    src = worker.RegionSource(bam_file)
    if refseq is not None:
        src.reader.set_reference(chrom, refseq)
    tally = worker.QnameTally()
    kept, laters = [], []
    starts = [s for _, s, _e in chunkloci_lst]
    groups = worker.group_chunks(chunkloci_lst)
    lo, hi = (min(starts), max(e for _, _s, e in chunkloci_lst) + (1 if phase else 0)) if starts else (None, None)
    decode = worker.choose_decode(decode, ctx, src.reader, chrom, lo, hi, len(groups), DEVICE_DECODE_MIN_BYTES)
    ctxs = [ctx] if (ctx2 is None or len(groups) == 1 or not hasattr(ctx, "call_chunks_submit")) else [ctx, ctx2]
    pins = worker.PinCache(ctx, enabled=len(groups) > 1)
    # `call` never needs the read bases as a stream: substituted bases are in the ops, and under a cs match the read
    # carries the reference allele of the site (cslib.py:22-29) — the decoder does not unpack them (seq=False) — and the
    # qualities travel as the decoder's parse pass leaves them: bitmap of the modal quality + exceptions, expanded on the
    # device (upload_compact).
    # --phase: the reference re-fetches [tpos, tpos + 1) at a site (caller.py:558), one position past a chunk that ends
    # at tpos: decode that position too, so a record that starts there is in the batch (it can only matter through a
    # shared query name)
    pending = None  # (context, chunk indices) of the call that is enqueued but not collected
    uploading = None  # (context, release) of the group whose upload has been enqueued but not waited for

    def finish(p):
        c, idx = p[0], p[1]
        rec, _log = c.call_chunks_collect(view=False) if len(ctxs) > 1 else p[2]
        tally.add(c.qname_seen())
        kept.append(rec)
        laters.append(min(starts[idx[-1] + 1:], default=None))

    lap = worker.Laps("call_region %s" % chrom)  # HIMUT_B200_WORKER_TIMING=1: where the host time of a contig goes
    if decode == "device":
        try:
            k = 0
            for idx in groups:
                loci = [chunkloci_lst[i] for i in idx]
                c = ctxs[k % len(ctxs)]  # never the context whose call is pending
                region = c.decode_region(src.reader, chrom, min(s for _, s, _e in loci), max(e for _, _s, e in loci) + (1 if phase else 0),
                                         ref=refseq)
                lap("device decode")
                if region.n_reads == 0:
                    continue
                k += 1
                table = region.chunk_table([(s, e) for _, s, e in loci], None if chunk_sets is None else [chunk_sets[i] for i in idx])
                if len(ctxs) > 1:
                    c.call_chunks_submit(table)
                    if pending is not None:
                        finish(pending)
                    pending = (c, idx)
                else:
                    finish((c, idx, c.call_chunks(table)))
                lap("submit + collect")
            if pending is not None:
                finish(pending)
            names = src.reader.qnames_blob(tally.seen) if want_names else None
        finally:
            src.close()
        kept = carry_som_seen(kept, laters)
        rec = np.concatenate(kept) if kept else np.zeros(0, abi.SITE_DTYPE)
        lap("merge")
        lap.report()
        return rec, tally.count(), names
    try:
        k = 0
        for idx, batch, cq, table, release in worker.pipelined_groups(src, chrom, chunkloci_lst, groups, chunk_sets, seq=False,
                                                                      pad=1 if phase else 0):
            lap("wait for decode")
            if batch.n_reads == 0:
                release()
                continue
            c = ctxs[k % len(ctxs)]
            k += 1
            pins.pin([cq.mask, cq.exc, batch.ops])
            lap("page-lock")
            if len(ctxs) > 1 and hasattr(c, "upload_wait"):
                # the copies of this group are enqueued before the previous group's are waited for (the copy engine goes
                # from one to the other), then the previous group's buffers go back to the decoder
                c.upload_compact(batch, cq, wait=False)
                if uploading is not None:
                    uploading[0].upload_wait()
                    uploading[1]()
                uploading = (c, release)
            else:
                c.upload_compact(batch, cq)
                release()  # everything is on the device: the decoder may reuse the buffers
            lap("upload")
            if len(ctxs) > 1:
                c.call_chunks_submit(table)
                if pending is not None:
                    finish(pending)
                pending = (c, idx)
            else:
                finish((c, idx, c.call_chunks(table)))
            lap("submit + collect")
        if uploading is not None:
            uploading[0].upload_wait()
            uploading[1]()
            uploading = None
        if pending is not None:
            finish(pending)
        lap("submit + collect")
        names = src.reader.qnames_blob(tally.seen) if want_names else None
    finally:
        if uploading is not None:  # an exception on the way: the copies must not outlive the decoder's buffers
            try:
                uploading[0].upload_wait()
            except Exception:
                pass
        pins.close()
        src.close()
        lap("unlock + close")
    kept = carry_som_seen(kept, laters)
    rec = np.concatenate(kept) if kept else np.zeros(0, abi.SITE_DTYPE)
    lap("merge")
    lap.report()
    return rec, tally.count(), names


def get_somatic_substitutions(
    chrom, bam_file, common_snps, panel_of_normals, chunkloci_lst, phase_set2hbit_lst, phase_set2hpos_lst,
    phase_set2hetsnp_lst, min_qv, min_mapq, qlen_lower_limit, qlen_upper_limit, min_sequence_identity, min_gq,
    min_bq, min_trim, max_mismatch_count, mismatch_window_size, md_threshold, min_ref_count, min_alt_count,
    min_hap_count, somatic_snv_prior, germline_snv_prior, germline_indel_prior, phase, non_human_sample,
    create_panel_of_normals, chrom2tsbs_lst, chrom2tsbs_log,
):
    ctx = worker.context()
    conf = (chrom, common_snps, panel_of_normals, chunkloci_lst, phase_set2hbit_lst, phase_set2hpos_lst,
            phase_set2hetsnp_lst, min_qv, min_mapq, qlen_lower_limit, qlen_upper_limit, min_sequence_identity,
            min_gq, min_bq, min_trim, max_mismatch_count, mismatch_window_size, md_threshold, min_ref_count,
            min_alt_count, min_hap_count, germline_snv_prior, phase, non_human_sample, create_panel_of_normals)
    chunk_sets = configure(ctx, *conf)
    ctx2 = None
    if len(worker.group_chunks(chunkloci_lst)) > 1 and hasattr(ctx, "call_chunks_submit"):
        ctx2 = worker.second_context()  # long contigs: two contexts alternate between decode groups
        configure(ctx2, *conf)
    rec, num_ccs, _ = call_region(ctx, bam_file, chrom, chunkloci_lst, chunk_sets, phase, ctx2=ctx2, refseq=worker.env_reference(chrom))
    chrom2tsbs_lst[chrom] = records.records_to_tsbs_lst(chrom, rec)
    chrom2tsbs_log[chrom] = [int(v) for v in _log_from_records(rec, num_ccs)]
    return int((rec["flags"] & abi.SITE_PL_TIE).astype(bool).sum())
