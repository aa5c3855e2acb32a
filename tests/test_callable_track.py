"""The callable-base track of `himut normcounts` on the CPU: the runs of the oracle's position loop
(tests/track_oracle.c, whose tallies are checked equal to the oracle's every time) against the reference's goldens — summed per trinucleotide bin they give back ref_tri2count / ccs_tri2count, summed over all
positions log[13] — the run-building rule against a plain restatement, and the drop-in worker writing one bedGraph per
contig under the oracle stand-in (HIMUT_B200_CALLABLE_TRACK)."""
import gzip
import json
import os

import numpy as np
import pytest

import cases
import parity
import standin_track
import track_oracle
from himut_b200 import abi, gtmodel, normcounts, synth, worker
from oracle import oracle

NORM_CASES = [n for n in cases.CASES if n.startswith("norm_")]
SWEEP = parity.load_random_sweep()


# ---- helpers (the GPU tests use them too) ----------------------------------------------------------------------
def tri_bins(ref):
    """tri_bin (oracle/himut_oracle.c) of every position of a contig: get_tri_context's bin, 32 = other"""
    s = np.frombuffer(ref.encode() if isinstance(ref, str) else bytes(ref), np.uint8)
    code = np.full(256, -1, np.int64)
    for ch, v in zip(b"ACGT", range(4)):
        code[ch] = v
    c = code[s]
    out = np.full(s.size, 32, np.int64)
    if s.size < 3:
        return out
    t0, t1, t2 = c[:-2], c[1:-1], c[2:]
    pur = (t1 == 0) | (t1 == 2)  # purine centre: reverse complement
    u0 = np.where(pur, np.where(t2 < 0, -1, 3 - t2), t0)
    u1 = np.where(pur, 3 - t1, t1)
    u2 = np.where(pur, np.where(t0 < 0, -1, 3 - t0), t2)
    ok = (t1 >= 0) & (u0 >= 0) & (u2 >= 0)
    out[1:-1] = np.where(ok, u0 * 8 + np.where(u1 == 3, 4, 0) + u2, 32)
    return out


def run_sums(runs, bins):
    """per bin: positions (ref_tri) and callable bases (ccs_tri) of the runs; and the callable bases of all of them"""
    n = (runs["end"].astype(np.int64) - runs["start"]).astype(np.int64)
    assert (n > 0).all()
    pos = np.repeat(runs["start"].astype(np.int64), n) + (np.arange(int(n.sum())) - np.repeat(np.cumsum(n) - n, n))
    val = np.repeat(runs["value"].astype(np.int64), n)
    b = bins[pos]
    return (np.bincount(b, minlength=abi.TRI_BINS), np.bincount(b, weights=val, minlength=abi.TRI_BINS).astype(np.int64),
            int(val.sum()))


def runs_from_dense(dense_per_chunk):
    """the run rule restated: per chunk (index, start, values of [start, end)), maximal ranges of equal non-zero value"""
    out = []
    for c, start, v in dense_per_chunk:
        i = 0
        while i < len(v):
            if v[i] == 0:
                i += 1
                continue
            j = i
            while j < len(v) and v[j] == v[i]:
                j += 1
            out.append((c, start + i, start + j, int(v[i])))
            i = j
    return np.array(out, abi.RUN_DTYPE) if out else np.zeros(0, abi.RUN_DTYPE)


def check_runs_shape(runs, chunk_table):
    """chunk order, then position order; inside the chunk; maximal (two runs of a chunk that touch differ in value)"""
    if not runs.size:
        return
    key = runs["chunk"].astype(np.int64) * (1 << 33) + runs["start"].astype(np.int64)
    assert (np.diff(key) > 0).all()
    ch = chunk_table[runs["chunk"]]
    assert (runs["start"] >= ch["start"]).all() and (runs["end"] <= ch["end"]).all()
    assert (runs["value"] >= 1).all()
    same = runs["chunk"][1:] == runs["chunk"][:-1]
    touch = same & (runs["start"][1:] == runs["end"][:-1])
    assert not (touch & (runs["value"][1:] == runs["value"][:-1])).any()


def tracked(params, batch, ref, table, common=None, pon=None, phase=None, alt_order=None):
    """the track oracle's tallies and runs; its tallies must be the oracle's own (it is the oracle's position loop with
    the track added)"""
    ao = None if alt_order is None else np.array(alt_order, np.uint8)
    res = track_oracle.normcounts_chunks_track(params, batch, ref, table, common, pon, phase, alt_order=ao)
    plain = oracle.normcounts_chunks(params, batch, ref, table, common, pon, phase, alt_order=ao)
    assert all(np.array_equal(a, b) for a, b in zip(plain[:3], res[:3])) and plain[3] == res[3]
    return res


def oracle_track(c, alt_order=None):
    return tracked(c["params"], c["batch"], c["ref"].encode(), c["chunk_table"], c["common"], c["pon"], c["phase"], alt_order)


def test_run_struct_layout():
    from himut_b200 import lib
    assert lib.load().hm_abi_sizeof(6) == abi.RUN_DTYPE.itemsize == 16


# ---- the oracle's runs against the goldens ----------------------------------------------------------------------
def _check_against(runs, ccs, rt, log, ref, chunk_table):
    check_runs_shape(runs, chunk_table)
    r_ref, r_ccs, total = run_sums(runs, tri_bins(ref))
    assert np.array_equal(r_ref, rt)
    assert np.array_equal(r_ccs, ccs)
    assert total == int(log[13])


@pytest.mark.parametrize("name", NORM_CASES)
def test_runs_sum_to_the_golden_tallies(name):
    fx = parity.load_golden(name)
    c = cases.build_case(name)
    e = fx["expected"]
    ccs, rt, log, _ties, runs = oracle_track(c, e["alt_order"])
    assert runs.size > 100
    _check_against(runs, parity.tri_dict_to_bins(e["ccs_tri2count"]), parity.tri_dict_to_bins(e["ref_tri2count"]),
                   e["log"], c["ref"], c["chunk_table"])


@pytest.mark.parametrize("seed", list(cases.RANDOM_NORM_SEEDS) + list(cases.RANDOM_LONG_NORM_SEEDS))
def test_runs_sum_to_the_random_sweep(seed):
    c = cases.random_case("norm", seed)
    if c is None:
        pytest.skip("no phase set")
    fx = SWEEP["norm"][str(seed)]
    ccs, rt, log, _ties, runs = oracle_track(c, fx["alt_order"])
    _check_against(runs, parity.tri_dict_to_bins(fx["ccs_tri2count"]), parity.tri_dict_to_bins(fx["ref_tri2count"]),
                   fx["log"], c["ref"], c["chunk_table"])


@pytest.mark.parametrize("seed", list(cases.RANDOM_CALL_SEEDS) + list(cases.RANDOM_LONG_CALL_SEEDS) + list(cases.RANDOM_DUPNAME_CALL_SEEDS))
def test_runs_sum_to_the_tallies_on_the_call_seeds(seed):
    """the sweep's `call` seeds have no normcounts golden: the runs against the oracle's own tallies of the same call"""
    c = cases.random_case("call", seed)
    if c is None:
        pytest.skip("no phase set")
    ccs, rt, log, _ties, runs = oracle_track(c)
    _check_against(runs, ccs, rt, log, c["ref"], c["chunk_table"])


def test_sweep_counts_81_seeds():
    assert len(SWEEP["call"]) + len(SWEEP["norm"]) == 81


# ---- overlapping chunk lists -------------------------------------------------------------------------------------
def overlap_case(contig_len=40_000, seed=7):
    d = synth.generate(contig_len, seed=seed, depth=30.0)
    p = gtmodel.make_params(**cases.call_args())
    loci = [(0, 12_000), (8_000, 20_000), (10_000, 11_000), (19_000, 40_000), (5_000, 30_000)]
    return d, p, loci, d.batch.chunk_table(loci)


def test_overlapping_chunks_count_a_position_once_per_chunk():
    d, p, loci, table = overlap_case()
    ccs, rt, log, _t, runs = tracked(p, d.batch, d.ref, table)
    _check_against(runs, ccs, rt, log, d.ref, table)
    # each chunk alone gives its own runs: the list's runs are theirs, chunk after chunk
    parts = []
    for i, l in enumerate(loci):
        one = tracked(p, d.batch, d.ref, d.batch.chunk_table([l]))[4]
        one["chunk"] = i
        parts.append(one)
    assert np.array_equal(np.concatenate(parts), runs)
    # positions in two chunks appear twice
    in_a = runs[(runs["chunk"] == 0) & (runs["end"] > 8_000)]
    in_b = runs[(runs["chunk"] == 1) & (runs["start"] < 12_000)]
    assert in_a.size and in_b.size


# ---- the run rule --------------------------------------------------------------------------------------------------
def test_run_rule_matches_a_dense_restatement():
    """the oracle's runs == the runs of the dense per-position values (value 0 = not counted) rebuilt here"""
    d, p, loci, table = overlap_case(seed=11)
    ccs, rt, log, _t, runs = tracked(p, d.batch, d.ref, table)
    dense = []
    for i, (s, e) in enumerate(loci):
        v = np.zeros(e - s, np.int64)
        for r in runs[runs["chunk"] == i]:
            v[r["start"] - s:r["end"] - s] = r["value"]
        dense.append((i, s, v))
    assert np.array_equal(runs_from_dense(dense), runs)
    # and the restatement itself on values built to test it: joins, breaks, chunk edges
    v = np.array([0, 3, 3, 3, 4, 4, 0, 0, 4, 4, 1, 0, 7], np.int64)
    got = runs_from_dense([(0, 100, v), (1, 113, np.array([7, 7, 0, 2], np.int64))])
    assert got.tolist() == [(0, 101, 104, 3), (0, 104, 106, 4), (0, 108, 110, 4), (0, 110, 111, 1), (0, 112, 113, 7),
                            (1, 113, 115, 7), (1, 116, 117, 2)]


# ---- the drop-in worker -----------------------------------------------------------------------------------------
GOLD2 = json.load(open(os.path.join(cases.GOLDEN_DIR, "cli_norm_phase.json")))


def _write_sites(path, per_contig):  # as tests/test_zz_pool.py writes them for the same golden
    text = ["##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tsynth\n"]
    for chrom, keys in per_contig:
        for k in keys.tolist():
            text.append("%s\t%d\t.\t%s\t%s\t.\tPASS\t.\tGT\t0/1\n" % (chrom, k >> 4, "ATGC"[(k >> 2) & 3], "ATGC"[k & 3]))
    with open(path, "wb") as f:
        f.write(gzip.compress("".join(text).encode()))


def _dropin(tmp, monkeypatch, track_dir):
    """get_callable_tricounts per contig of tests/golden/cli_norm_phase.json, as the pool of `himut normcounts` calls it"""
    from himut_b200 import bamio
    data = cases.cli_dataset(None)
    bam = os.path.join(tmp, "synth.bam")
    bamio.write_batches_bam(bam, [(c, n, d.batch) for c, n, d in data])
    sets = [(c,) + cases.site_sets_from_synth(d, 40 + i) for i, (c, _n, d) in enumerate(data)]
    common, pon = os.path.join(tmp, "common.vcf.bgz"), os.path.join(tmp, "pon.vcf.bgz")
    _write_sites(common, [(c, k) for c, k, _ in sets])
    _write_sites(pon, [(c, k) for c, _, k in sets])
    ctx = standin_track.TrackOracleContext()
    monkeypatch.setattr(worker, "context", lambda: ctx)
    plain = worker.RegionSource.batch
    monkeypatch.setattr(worker.RegionSource, "batch",
                        lambda self, chrom, loci, phase_sets=None, seq=True, **kw: plain(self, chrom, loci, phase_sets, seq=True, **kw))
    if track_dir is None:
        monkeypatch.delenv(normcounts.CALLABLE_TRACK_ENV, raising=False)
    else:
        monkeypatch.setenv(normcounts.CALLABLE_TRACK_ENV, track_dir)
    a = dict(gtmodel.DEFAULT_CALL_ARGS)
    qlo, qhi, md = GOLD2["normcounts"]["thresholds"]
    by = {c: (n, d) for c, n, d in data}
    ccs, rt, log = {}, {}, {}
    for c in GOLD2["normcounts"]["contigs"]:
        n, d = by[c]
        normcounts.get_callable_tricounts(
            c, d.ref.decode(), bam, common, pon, [(c, s, e) for s, e in cases.chunkloci(0, n)], {}, {}, {},
            a["min_qv"], a["min_mapq"], a["min_trim"], qlo, qhi, a["min_sequence_identity"], a["min_gq"], a["min_bq"],
            a["mismatch_window"], a["max_mismatch_count"], a["min_ref_count"], a["min_alt_count"], a["min_hap_count"], md,
            1 / (10 ** 6), a["germline_snv_prior"], 1 / (10 ** 4), False, False, ccs, rt, log)
    return by, ccs, rt, log


def _read_bedgraph(path):
    rows = [l.split("\t") for l in open(path).read().splitlines()]
    return rows


def test_dropin_writes_one_bedgraph_per_contig(tmp_path, monkeypatch):
    track = tmp_path / "track"
    track.mkdir()
    by, ccs, rt, log = _dropin(str(tmp_path), monkeypatch, str(track))
    contigs = GOLD2["normcounts"]["contigs"]
    assert sorted(os.listdir(track)) == sorted("%s.callable.bedgraph" % c for c in contigs)
    tot_ref = np.zeros(abi.TRI_BINS, np.int64)
    tot_ccs = np.zeros(abi.TRI_BINS, np.int64)
    for c in contigs:
        rows = _read_bedgraph(str(track / ("%s.callable.bedgraph" % c)))
        assert rows and all(r[0] == c and len(r) == 4 for r in rows)
        runs = np.array([(0, int(s), int(e), int(v)) for _c, s, e, v in rows], abi.RUN_DTYPE)
        r_ref, r_ccs, total = run_sums(runs, tri_bins(by[c][1].ref))
        tot_ref += r_ref
        tot_ccs += r_ccs
        assert total == log[c][13]
    exp = GOLD2["normcounts"]["tri"]
    assert {t: [int(tot_ref[i]), int(tot_ccs[i])] for i, t in enumerate(normcounts.TRI_LST)} == exp
    # with the variable unset: no file, the same results
    track2 = tmp_path / "unset"
    track2.mkdir()
    monkeypatch.chdir(track2)
    _by, ccs2, rt2, log2 = _dropin(str(tmp_path), monkeypatch, None)
    assert os.listdir(track2) == []
    assert (ccs2, rt2, log2) == (ccs, rt, log)
    assert {c: log2[c] for c in contigs} == GOLD2["normcounts"]["log"]
