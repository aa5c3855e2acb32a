"""`himut call` over a whole genome on N GPUs: chunk runs sharded over ranks (SURVEY.md §8e, BASELINE configs[2]).

The reference parallelises with one pool process per chromosome (src/himut/caller.py:766-810) over util.chunkloci's
200 kb chunks (src/himut/util.py:119-132); a single contig runs on one core whatever --threads says.  Here the unit
is a *run* of consecutive chunks of one contig: long contigs are cut into several runs so that eight GPUs get even
shares of a genome whose largest contig is 8 % of it, short contigs stay whole.  Adjacent chunks stay together, so
the som_seen carry (caller.py:243,347; bamlib.py:77) is the worker's own inside a run; between two runs of a contig it
is replayed at the merge from the records themselves, exactly as the worker replays it between its decode groups
(caller.carry_som_seen).  No data-path collective exists: every rank runs the worker's device path on its runs, then
the records, the counts of distinct query names (for a split contig: the names, m.num_ccs counts them per contig) and
a few statistics are gathered on rank 0, which builds the reference's per-contig tuple lists and log vectors for its
unchanged writers.

Launch: one process per GPU under torchrun (`torch.distributed` initialised, NCCL on GPUs, gloo in the CPU tests), or
a single process (world size 1).  `python -m himut_b200.genome --help` is the command-line form.
"""
import os
import time

import numpy as np

from . import abi, caller, fasta, records, shard, worker


class Run:
    """consecutive chunks [lo, hi) of one contig's chunk list"""
    __slots__ = ("index", "chrom", "lo", "hi", "weight", "rank")

    def __init__(self, index, chrom, lo, hi, weight):
        self.index, self.chrom, self.lo, self.hi, self.weight, self.rank = index, chrom, lo, hi, weight, 0

    def __repr__(self):
        return "Run(%d, %s[%d:%d], w=%d, rank=%d)" % (self.index, self.chrom, self.lo, self.hi, self.weight, self.rank)


def plan_runs(chrom2chunkloci, world, pieces_per_rank=4, chunk_weight=None, how="contiguous"):
    """cut the genome's chunk lists into runs (consecutive chunks of one contig) and assign them to ranks.
    Deterministic: every rank computes the same plan.  Weight of a chunk: its reference span, or
    chunk_weight(chrom, start, end).

    how="contiguous" (default): the chunks of all contigs, in contig order, are cut into `world` consecutive pieces
      of equal weight (to within one chunk); a rank's runs are the intersections of its piece with the contigs, so a
      rank sees at most two partial contigs and the loads differ by at most one 200 kb chunk.
    how="lpt": every contig is cut into runs no heavier than total / (world * pieces_per_rank) (contigs lighter than
      that stay whole) and the runs go to ranks longest-processing-time first (shard.lpt_assign: heaviest run to the
      least loaded rank, ties to the lower rank) — for weights that are not known to be even along a contig."""
    w = chunk_weight or (lambda c, s, e: max(int(e) - int(s), 1))
    weights = {c: [w(*x) for x in lst] for c, lst in chrom2chunkloci.items()}
    total = sum(sum(v) for v in weights.values())
    world = max(world, 1)
    runs = []
    if how == "contiguous":
        rank, acc = 0, 0
        for chrom, lst in chrom2chunkloci.items():
            lo = 0
            for i, wi in enumerate(weights[chrom]):
                # the chunk goes to the rank in whose share its midpoint falls
                mid_rank = min(world - 1, int((acc + wi / 2.0) * world / total)) if total else 0
                if mid_rank != rank:
                    if i > lo:
                        runs.append(Run(len(runs), chrom, lo, i, sum(weights[chrom][lo:i])))
                        runs[-1].rank = rank
                    lo, rank = i, mid_rank
                acc += wi
            if len(lst) > lo:
                runs.append(Run(len(runs), chrom, lo, len(lst), sum(weights[chrom][lo:])))
                runs[-1].rank = rank
        return runs
    limit = total if world <= 1 else max(1, total // (world * max(1, pieces_per_rank)))
    for chrom, lst in chrom2chunkloci.items():
        ws = weights[chrom]
        if not lst:
            continue
        tot = sum(ws)
        n_pieces = min(len(ws), max(1, -(-tot // limit)))  # pieces of about equal weight, cut at chunk edges
        cum, acc = [], 0
        for wi in ws:
            acc += wi
            cum.append(acc)
        bounds, i = [0], 0
        for k in range(1, n_pieces):
            target = tot * k / n_pieces
            while i < len(ws) - 1 and cum[i] < target:
                i += 1
            cut = max(i + 1, bounds[-1] + 1)
            if cut < len(ws):
                bounds.append(cut)
        bounds.append(len(ws))
        for lo, hi in zip(bounds, bounds[1:]):
            runs.append(Run(len(runs), chrom, lo, hi, sum(ws[lo:hi])))
    assign = shard.lpt_assign({r.index: r.weight for r in runs}, world)
    for r in runs:
        r.rank = assign[r.index]
    return runs


def imbalance(runs, world):
    """max / mean of the per-rank weight (1.0 = perfectly even)"""
    load = [0] * max(world, 1)
    for r in runs:
        load[r.rank] += r.weight
    mean = sum(load) / len(load)
    return (max(load) / mean) if mean else 1.0


def _dist():
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist
    except Exception:
        pass
    return None


def call_genome(bam_file, chrom2chunkloci, args, phase_tables=None, common_snps=None, panel_of_normals=None, pieces_per_rank=4,
                ctx=None, ref=None):
    """`himut call` over every contig of chrom2chunkloci (contig -> its chunkloci list, as util.load_loci /
    vcflib.load_phased_hetsnps build it), sharded over the ranks of the initialised process group.

    args: the worker's scalar arguments by name (gtmodel.DEFAULT_CALL_ARGS keys + phase / non_human_sample /
          create_panel_of_normals);  phase_tables: contig -> (hbit, hpos, hetsnp dicts) in --phase mode.
    ref: a FASTA of the reference the reads were aligned to, for records with neither cs:Z nor MD:Z (each run reads
    its contig from it).
    Returns on rank 0 (chrom2tsbs_lst, chrom2tsbs_log, stats) — the dictionaries the reference's dump_call_log /
    dump_sbs / dump_phased_sbs take (vcflib.py:820-1060) — and (None, None, stats) on the other ranks."""
    dist = _dist()
    rank = dist.get_rank() if dist else 0
    world = dist.get_world_size() if dist else 1
    runs = plan_runs(chrom2chunkloci, world, pieces_per_rank)
    per_contig = {}
    for r in runs:
        per_contig.setdefault(r.chrom, []).append(r)
    own_ctx = ctx is None
    ctx = ctx or worker.context()
    phase = bool(args.get("phase"))
    local, t0, my_weight = [], time.perf_counter(), 0
    ref_contig = (None, None)
    for r in runs:
        if r.rank != rank:
            continue
        chunks = chrom2chunkloci[r.chrom][r.lo:r.hi]
        hbit, hpos, hetsnp = (phase_tables or {}).get(r.chrom, ({}, {}, {}))
        conf = (r.chrom, common_snps, panel_of_normals, chunks, hbit, hpos, hetsnp, args["min_qv"], args["min_mapq"],
                args["qlen_lower_limit"], args["qlen_upper_limit"], args["min_sequence_identity"], args["min_gq"], args["min_bq"],
                args["min_trim"], args["max_mismatch_count"], args["mismatch_window"], args["md_threshold"], args["min_ref_count"],
                args["min_alt_count"], args["min_hap_count"], args["germline_snv_prior"], phase, bool(args.get("non_human_sample")),
                bool(args.get("create_panel_of_normals")))
        chunk_sets = caller.configure(ctx, *conf)
        ctx2 = None
        if own_ctx and len(worker.group_chunks(chunks)) > 1:  # long runs: two contexts alternate between decode groups
            ctx2 = worker.second_context()
            caller.configure(ctx2, *conf)
        split = len(per_contig[r.chrom]) > 1
        if ref and r.chrom != ref_contig[0]:  # read once per contig: its runs on this rank reuse it, uploads included
            ref_contig = (r.chrom, fasta.load_contig(ref, r.chrom))
        refseq = ref_contig[1] if ref else None
        rec, num_ccs, names = caller.call_region(ctx, bam_file, r.chrom, chunks, chunk_sets, phase, want_names=split, ctx2=ctx2,
                                                 refseq=refseq)
        local.append((r.index, rec, num_ccs, names))
        my_weight += r.weight
    seconds = time.perf_counter() - t0
    # the only cross-rank step: results to rank 0 (records, name blobs of split contigs), a few statistics to everyone
    if dist:
        bucket = [None] * world if rank == 0 else None
        dist.gather_object(local, bucket, dst=0)
        stat = shard.all_reduce_sum(np.asarray([my_weight, sum(x[1].size for x in local), int(seconds * 1e6)], np.int64),
                                    device=_stat_device(dist))
        tmax = shard.all_reduce_max(np.asarray([int(seconds * 1e6)], np.int64), device=_stat_device(dist))
    else:
        bucket = [local]
        stat = np.asarray([my_weight, sum(x[1].size for x in local), int(seconds * 1e6)], np.int64)
        tmax = np.asarray([int(seconds * 1e6)], np.int64)
    stats = {"world": world, "runs": len(runs), "split_contigs": sum(1 for v in per_contig.values() if len(v) > 1),
             "imbalance_max_over_mean": imbalance(runs, world), "records": int(stat[1]),
             "rank_seconds_max": float(tmax[0]) * 1e-6, "rank_seconds_mean": float(stat[2]) * 1e-6 / world}
    if rank != 0:
        return None, None, stats
    by_index = {}
    for part in bucket:
        for idx, rec, num_ccs, names in part:
            by_index[idx] = (rec, num_ccs, names)
    chrom2tsbs_lst, chrom2tsbs_log = {}, {}
    for chrom, rs in per_contig.items():
        rs = sorted(rs, key=lambda r: r.lo)
        lst = chrom2chunkloci[chrom]
        parts = [by_index[r.index][0] for r in rs]
        laters = [min((s for _c, s, _e in lst[r.hi:]), default=None) for r in rs]
        rec = np.concatenate(caller.carry_som_seen(parts, laters)) if parts else np.zeros(0, abi.SITE_DTYPE)
        if len(rs) == 1:
            num_ccs = by_index[rs[0].index][1]
        else:  # distinct query names over the whole contig (m.num_ccs, caller.py:318-320)
            seen = set()
            for r in rs:
                seen.update(n for n in by_index[r.index][2].split(b"\n") if n)
            num_ccs = len(seen)
        chrom2tsbs_lst[chrom] = records.records_to_tsbs_lst(chrom, rec)
        chrom2tsbs_log[chrom] = [int(v) for v in caller._log_from_records(rec, num_ccs)]
    return chrom2tsbs_lst, chrom2tsbs_log, stats


def _stat_device(dist):
    """tensors of an NCCL group live on the rank's GPU"""
    if dist.get_backend() == "nccl":
        import torch
        return torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    return None


def chunkloci(chrom, length, chunk=200_000):
    """util.chunkloci for a whole contig (src/himut/util.py:119-132)"""
    if length <= chunk:
        return [(chrom, 0, length)]
    starts = list(range(chunk, length, chunk))
    out = [(chrom, 1, chunk)]
    for i, s in enumerate(starts[:-1]):
        out.append((chrom, s, starts[i + 1]))
    out.append((chrom, starts[-1], length - 2))
    return out


def main(argv=None):
    """python -m himut_b200.genome -i in.bam -o out.vcf [--non_human_sample ...]: every contig of the BAM, all GPUs
    of the job; rank 0 writes the VCF (+ single-molecule twin) and himut.log with the mirrors of the reference's
    writers (vcfio.dump_sbs, the log in dump_call_log's format)"""
    import argparse
    from . import bamdec, bamlib, gtmodel, vcfio
    ap = argparse.ArgumentParser(prog="himut_b200.genome")
    ap.add_argument("-i", "--bam", required=True)
    ap.add_argument("-o", "--vcf", required=True)
    ap.add_argument("--common_snps")
    ap.add_argument("--panel_of_normals")
    ap.add_argument("--non_human_sample", action="store_true")
    ap.add_argument("--pieces_per_rank", type=int, default=4)
    ap.add_argument("--ref", help="FASTA of the reference the reads were aligned to: decodes records with neither cs:Z nor MD:Z")
    a = ap.parse_args(argv)
    if "RANK" in os.environ and "WORLD_SIZE" in os.environ and int(os.environ["WORLD_SIZE"]) > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dist.init_process_group(backend)
    nb = bamdec.NativeBam(a.bam)
    contigs = list(zip(nb.references, nb.lengths))
    nb.close()
    tname2tsize = dict(contigs)
    lo, hi, md = bamlib.get_thresholds(a.bam, [c for c, _ in contigs], tname2tsize)
    args = dict(gtmodel.DEFAULT_CALL_ARGS, qlen_lower_limit=lo, qlen_upper_limit=hi, md_threshold=md,
                non_human_sample=a.non_human_sample)
    loci = {c: chunkloci(c, n) for c, n in contigs}
    lst, log, stats = call_genome(a.bam, loci, args, common_snps=a.common_snps, panel_of_normals=a.panel_of_normals,
                                  pieces_per_rank=a.pieces_per_rank, ref=a.ref)
    if lst is not None:
        from .natsort_compat import natsorted
        chroms = natsorted(list(lst))
        header = "##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tsample"
        vcfio.dump_sbs(a.vcf, header, chroms, lst)
        with open("himut.log", "w") as f:
            for c in chroms:
                f.write("%s\t%s\n" % (c, "\t".join(str(v) for v in log[c])))
        print("himut_b200.genome: %d contigs, %d rows, %s" % (len(chroms), sum(len(v) for v in lst.values()), stats))
    d = _dist()
    if d:
        d.barrier()
        d.destroy_process_group()


if __name__ == "__main__":
    main()
