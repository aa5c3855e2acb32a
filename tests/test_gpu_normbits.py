"""The bit-vector integer pass of `himut normcounts` (himut_b200/csrc/normbits.cuh: k_norm_prep + k_norm_bits) on its
edges, against the CPU oracle; and on the same 300 kb batch the single pass k_norm_tiles_tma that genotypes every
column exactly where the parameters lie outside the certified domain.  GPU."""
import numpy as np
import pytest

import cases
from himut_b200 import gtmodel, synth
from oracle import oracle

pytestmark = pytest.mark.gpu


def run(ctx, p, d, loci):
    chunks = d.batch.chunk_table(loci)
    ctx.set_params(p)
    ctx.set_site_sets()
    ctx.upload(d.batch)
    g = ctx.normcounts_chunks(d.ref, chunks)
    o = oracle.normcounts_chunks(p, d.batch, d.ref, chunks)
    return g, o


def same(g, o):
    return np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1]) and list(g[2]) == list(o[2]) and g[3] == o[3]


def test_bits_and_single_pass_on_300_kb(ctx):
    d = synth.generate(300_000, seed=41)
    p = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
    loci = cases.chunkloci(0, 300_000)
    g, o = run(ctx, p, d, loci)
    assert same(g, o)
    names = [n for n, _ in ctx.last_kernel_times()]
    assert "k_norm_prep" in names and "k_norm_bits" in names and "k_norm_tiles_tma" not in names
    # the bit-vector pass is deterministic: exactly these positions reach the exact pass
    assert ctx.last_norm_exact_sites() == 2771
    # min_bq 0 lies outside the certified domain: the single pass genotypes every column
    p = gtmodel.make_params(**cases.call_args(min_bq=0))
    g, o = run(ctx, p, d, loci)
    assert same(g, o)
    names = [n for n, _ in ctx.last_kernel_times()]
    assert "k_norm_tiles_tma" in names and "k_norm_bits" not in names


@pytest.mark.parametrize("over", [dict(max_mismatch_count=2), dict(max_mismatch_count=1, mismatch_window=40),
                                  dict(mismatch_window=0), dict(min_trim=0.2), dict(min_trim=0.0),
                                  dict(min_bq=20), dict(min_bq=94), dict(min_qv=93), dict(min_mapq=61),
                                  dict(md_threshold=20), dict(md_threshold=31.5), dict(min_ref_count=31)])
def test_parameters(ctx, over):
    d = synth.generate(150_000, seed=42)
    p = gtmodel.make_params(**cases.call_args(**over))
    g, o = run(ctx, p, d, [(0, 70_001), (70_001, 150_000)])
    assert same(g, o)


def test_reads_of_several_segments(ctx):
    """reads of 40 - 60 kb: k_norm_prep walks a read in segments of 8192 query bases; words of cal bits that two
    segments share, match runs and mismatch windows that cross a segment border"""
    d = synth.generate(400_000, seed=43, read_len_min=40_000, read_len_max=60_000, depth=20.0)
    p = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
    g, o = run(ctx, p, d, cases.chunkloci(0, 400_000))
    assert same(g, o)
    assert ctx.last_norm_exact_sites() < 40_000
    # no mismatch at all for long stretches: match runs longer than a segment
    d = synth.generate(300_000, seed=47, read_len_min=20_000, read_len_max=30_000, depth=15.0, sub_err_rate=0.0, indel_rate=0.0,
                       somatic_rate=0.0, het_rate=2e-5, hom_rate=1e-5)
    g, o = run(ctx, p, d, cases.chunkloci(0, 300_000))
    assert same(g, o)


def test_dense_ops(ctx):
    """reads with hundreds of cs ops (more than a warp stages): exact pass for their span; and just below that bound"""
    for rate, seed in ((0.02, 44), (0.004, 45)):
        d = synth.generate(120_000, seed=seed, indel_rate=rate)
        p = gtmodel.make_params(**cases.call_args(min_sequence_identity=0.5))
        g, o = run(ctx, p, d, [(0, 120_000)])
        assert same(g, o)


def test_chunks_off_the_grid(ctx):
    """chunk borders inside a 32-position word and inside a 1024-position span, one-position chunks, a chunk past the
    last read, overlapping chunks"""
    d = synth.generate(100_000, seed=46)
    p = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
    loci = [(0, 1), (1, 33), (33, 1023), (1023, 1025), (1025, 50_000), (49_000, 51_017), (51_017, 99_999), (99_999, 100_000)]
    g, o = run(ctx, p, d, loci)
    assert same(g, o)
    for l in loci:
        g, o = run(ctx, p, d, [l])
        assert same(g, o), l


def test_phase_and_sets_cases_on_the_bit_path(ctx):
    for name in ("norm_phase", "norm_config3_phase_sets", "norm_adversarial", "norm_sets"):
        if name not in cases.CASES:
            continue
        c = cases.build_case(name)
        ctx.set_params(c["params"])
        ctx.set_site_sets(c["common"], c["pon"])
        if c["phase"] is not None:
            ctx.set_phase_sets(c["phase"])
        ctx.upload(c["batch"])
        g = ctx.normcounts_chunks(c["ref"].encode(), c["chunk_table"])
        o = oracle.normcounts_chunks(c["params"], c["batch"], c["ref"].encode(), c["chunk_table"], c["common"], c["pon"], c["phase"])
        assert same(g, o), name
        assert "k_norm_bits" in [n for n, _ in ctx.last_kernel_times()], name


@pytest.mark.parametrize("over", [dict(), dict(min_bq=20), dict(min_bq=94), dict(min_bq=60, min_trim=0.05), dict(min_qv=92)])
def test_compact_upload_takes_the_bits_from_the_bitmap(ctx, over):
    """a batch uploaded as modal bitmap + exceptions (what the workers upload): where every exception of a read lies
    below min_bq the bit "BQ >= min_bq" is the bitmap's and the quality sum is the one taken at expansion; a read with
    an exception at or above min_bq goes through its quality bytes; both must equal the plain upload and the oracle"""
    from himut_b200 import bamdec
    d = synth.generate(250_000, seed=48, read_len_min=9_000, read_len_max=21_000)
    p = gtmodel.make_params(**cases.call_args(**over))
    loci = cases.chunkloci(0, 250_000)
    chunks = d.batch.chunk_table(loci)
    o = oracle.normcounts_chunks(p, d.batch, d.ref, chunks)
    cq = bamdec.compact_bq(d.batch, threads=2)
    ctx.set_params(p)
    ctx.set_site_sets()
    ctx.upload_compact(d.batch, cq)
    g = ctx.normcounts_chunks(d.ref, chunks)
    assert same(g, o)
    rec, log = ctx.call_chunks(chunks)  # the expanded stream is still what `call` reads
    o_rec, o_log = oracle.call_chunks(p, d.batch, chunks)
    assert list(log) == list(o_log)
