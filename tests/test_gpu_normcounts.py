"""Parity of the CUDA callable-base half of `himut normcounts` (through the C ABI) with the CPU
oracle and with the reference's own outputs (golden fixtures).  Needs a B200: `pytest -m gpu`."""
import numpy as np
import pytest

import cases
import parity
from himut_b200 import abi, gtmodel, synth
from oracle import oracle

pytestmark = pytest.mark.gpu
NORM_CASES = [n for n in cases.CASES if n.startswith("norm_")]


def run_gpu(ctx, c):
    ctx.set_params(c["params"])
    ctx.set_site_sets(c["common"], c["pon"])
    if c["phase"] is not None:
        ctx.set_phase_sets(c["phase"])
    ctx.upload(c["batch"])
    return ctx.normcounts_chunks(c["ref"].encode(), c["chunk_table"])


@pytest.mark.parametrize("name", NORM_CASES)
def test_normcounts_matches_oracle(ctx, name):
    c = cases.build_case(name)
    ccs, rt, log, ties = run_gpu(ctx, c)
    o_ccs, o_rt, o_log, o_ties = oracle.normcounts_chunks(c["params"], c["batch"], c["ref"].encode(), c["chunk_table"],
                                                          c["common"], c["pon"], c["phase"])
    assert np.array_equal(ccs, o_ccs)
    assert np.array_equal(rt, o_rt)
    assert list(log) == list(o_log)
    assert ties == o_ties


@pytest.mark.parametrize("name", NORM_CASES)
def test_normcounts_matches_reference(ctx, name):
    """the golden run iterated the alt set in a hash-seed order; positions where that order can
    matter are the flagged ties, so the comparison is exact whenever the fixture has none"""
    c = cases.build_case(name)
    fx = parity.load_golden(name)
    e = fx["expected"]
    canonical = [[a for a in range(4) if a != r] for r in range(4)]
    ccs, rt, log, ties = run_gpu(ctx, c)
    if e["alt_order"] != canonical and ties:
        o = oracle.normcounts_chunks(c["params"], c["batch"], c["ref"].encode(), c["chunk_table"], c["common"], c["pon"],
                                     c["phase"], alt_order=np.array(e["alt_order"], np.uint8))
        if not (np.array_equal(o[0], ccs) and list(o[2]) == list(log)):
            pytest.skip("%d alt ties: the reference's own result depends on PYTHONHASHSEED here" % ties)
    assert np.array_equal(ccs, parity.tri_dict_to_bins(e["ccs_tri2count"]))
    assert np.array_equal(rt, parity.tri_dict_to_bins(e["ref_tri2count"]))
    assert [int(v) for v in log] == e["log"]


def test_normcounts_one_megabase(ctx):
    d = synth.generate(1_000_000, seed=31)
    p = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
    chunks = d.batch.chunk_table(cases.chunkloci(0, 1_000_000))
    ctx.set_params(p)
    ctx.set_site_sets()
    ctx.upload(d.batch)
    ccs, rt, log, ties = ctx.normcounts_chunks(d.ref, chunks)
    o = oracle.normcounts_chunks(p, d.batch, d.ref, chunks)
    assert np.array_equal(ccs, o[0]) and np.array_equal(rt, o[1]) and list(log) == list(o[2]) and ties == o[3]
    assert int(log[13]) > 20_000_000


def test_normcounts_additive_over_chunks(ctx):
    """property: bins and counters of a chunk list are the sums over its chunks"""
    d = synth.generate(100_000, seed=32)
    p = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
    ctx.set_params(p)
    ctx.set_site_sets()
    ctx.upload(d.batch)
    loci = [(0, 30_000), (30_000, 65_001), (65_001, 100_000)]
    whole = ctx.normcounts_chunks(d.ref, d.batch.chunk_table(loci))
    parts = [ctx.normcounts_chunks(d.ref, d.batch.chunk_table([l])) for l in loci]
    assert np.array_equal(whole[0], sum(x[0] for x in parts))
    assert np.array_equal(whole[1], sum(x[1] for x in parts))
    assert list(whole[2][1:]) == list(sum(x[2] for x in parts)[1:])  # num_ccs is a distinct count, not additive


def test_normcounts_chunk_with_a_negative_start(ctx):
    """a fetch window that starts before the contig: the bit-vector pass works on the absolute 1024-position grid and
    leaves such a call to the single pass, whose tiles are chunk-relative; positions below 0 count for nothing"""
    d = synth.generate(100_000, seed=37)
    p = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
    chunks = d.batch.chunk_table([(-500, 40_000), (40_000, 100_000)])
    ctx.set_params(p)
    ctx.set_site_sets()
    ctx.upload(d.batch)
    g = ctx.normcounts_chunks(d.ref, chunks)
    o = oracle.normcounts_chunks(p, d.batch, d.ref, chunks)
    assert np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1]) and list(g[2]) == list(o[2]) and g[3] == o[3]
    assert "k_norm_tiles_tma" in [n for n, _ in ctx.last_kernel_times()]


@pytest.mark.parametrize("over", [dict(min_gq=60), dict(min_gq=99), dict(min_gq=0, germline_snv_prior=0.3),
                                  dict(min_bq=1, min_gq=35, md_threshold=25), dict(min_ref_count=40)])
def test_normcounts_certification_edges(ctx, over):
    """parameters that push many pure positions out of the certified domain (or make every one fail a gate):
    whatever the integer pass cannot decide must come back through the exact pass with the oracle's answer"""
    d = synth.generate(200_000, seed=33)
    p = gtmodel.make_params(**cases.call_args(**over))
    chunks = d.batch.chunk_table(cases.chunkloci(0, 200_000))
    ctx.set_params(p)
    ctx.set_site_sets()
    ctx.upload(d.batch)
    g = ctx.normcounts_chunks(d.ref, chunks)
    o = oracle.normcounts_chunks(p, d.batch, d.ref, chunks)
    assert np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1]) and list(g[2]) == list(o[2]) and g[3] == o[3]


@pytest.mark.parametrize("slots", [None, "64"])
def test_normcounts_deep_pileup(ctx, slots, monkeypatch):
    """400x: more than 255 reads per 1024-position span (the 8-bit bit-sliced counters of k_norm_bits would overflow:
    the whole span goes to the exact pass) and more reads per position than the entry table has slots (512 at most;
    64 when HIMUT_B200_SITE_SLOTS forces it): the reduce computes the slots beyond the table itself"""
    if slots is not None:
        monkeypatch.setenv("HIMUT_B200_SITE_SLOTS", slots)  # read at upload
    d = synth.generate(30_000, seed=34, depth=400.0)
    p = gtmodel.make_params(**cases.call_args(md_threshold=1000))
    chunks = d.batch.chunk_table([(0, 12_345), (12_345, 30_000)])
    ctx.set_params(p)
    ctx.set_site_sets()
    ctx.upload(d.batch)
    g = ctx.normcounts_chunks(d.ref, chunks)
    assert ctx.last_norm_exact_sites() > 25_000
    o = oracle.normcounts_chunks(p, d.batch, d.ref, chunks)
    assert np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1]) and list(g[2]) == list(o[2]) and g[3] == o[3]
    # the same data through `call`: deep pileups there too
    rec, log = ctx.call_chunks(chunks)
    o_rec, o_log = oracle.call_chunks(p, d.batch, chunks)
    ok, why = parity.records_equal(rec, o_rec)
    assert ok, why
    assert list(log) == list(o_log)


@pytest.mark.parametrize("depth", [60.0, 100.0])
def test_normcounts_deeper_samples(ctx, depth):
    """60x / 100x: the entry slots of the exact pass follow the depth, the bit-sliced counters hold up to 255 reads"""
    d = synth.generate(60_000, seed=36, depth=depth)
    p = gtmodel.make_params(**cases.call_args(md_threshold=1000))
    chunks = d.batch.chunk_table([(0, 30_000), (30_000, 60_000)])
    ctx.set_params(p)
    ctx.set_site_sets()
    ctx.upload(d.batch)
    g = ctx.normcounts_chunks(d.ref, chunks)
    o = oracle.normcounts_chunks(p, d.batch, d.ref, chunks)
    assert np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1]) and list(g[2]) == list(o[2]) and g[3] == o[3]
