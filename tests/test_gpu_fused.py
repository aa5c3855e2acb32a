"""The fused `himut call` device path (csrc/callfused.cuh) against the oracle on the shapes that exercise its own
machinery — several sort tiles per chunk, more distinct positions per tile than fit in shared memory, op lists longer
than a warp stages, the site-buffer overflow retry, reads that fail the QV gate (k_call_pairs emits no candidate for
them) — and the first version of the path (HIMUT_B200_CALL_V1=1), which stays as the route for chunk spans of 2^27
and more, on every fixed case.  GPU."""
import numpy as np
import pytest

import cases
import parity
from himut_b200 import gtmodel, lib, synth
from oracle import oracle

pytestmark = pytest.mark.gpu
CALL_CASES = [n for n in cases.CASES if n.startswith("call_")]


def _same_as_oracle(ctx, p, batch, chunks, common=None, pon=None, phase=None, path=2, full=None):
    """full: the batch with its base stream when `batch` comes without (the oracle reads the bases)"""
    ctx.set_params(p)
    ctx.set_site_sets(common, pon)
    if phase is not None:
        ctx.set_phase_sets(phase)
    rec, log = ctx.call_batch(batch, chunks)
    assert ctx.last_call_path() == path
    o_rec, o_log = oracle.call_chunks(p, full if full is not None else batch, chunks, common, pon, phase)
    ok, why = parity.records_equal(rec, o_rec)
    assert ok, why
    assert list(log) == list(o_log)
    return rec, log


@pytest.mark.parametrize("name", CALL_CASES)
def test_first_version_still_matches(name, monkeypatch):
    monkeypatch.setenv("HIMUT_B200_CALL_V1", "1")
    c = cases.build_case(name)
    with lib.Context(0) as ctx:
        _same_as_oracle(ctx, c["params"], c["batch"], c["chunk_table"], c["common"], c["pon"], c["phase"], path=1)


def test_fused_is_the_default(ctx):
    c = cases.build_case("call_basic")
    _same_as_oracle(ctx, c["params"], c["batch"], c["chunk_table"], c["common"], c["pon"], c["phase"], path=2)
    names = [n for n, _ms in ctx.last_kernel_times()]
    assert "k_call_scan" in names and "k_call_pairs" in names and not any(n.startswith("cub") for n in names)


def test_one_chunk_of_several_tiles(ctx):
    """a 600 kb contig as a single chunk: five 2^17-position sort tiles share the chunk's key segment"""
    d = synth.generate(600_000, seed=31)
    p = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
    _same_as_oracle(ctx, p, d.batch, d.batch.chunk_table([(0, 600_000)]))
    _same_as_oracle(ctx, p, d.batch.without_seq(), d.batch.chunk_table([(0, 600_000)]), full=d.batch)


def test_site_buffer_overflow_retries(ctx, monkeypatch):
    monkeypatch.setenv("HIMUT_B200_SITE_CAP", "8")
    d = synth.generate(120_000, seed=77)
    p = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
    rec, _ = _same_as_oracle(ctx, p, d.batch, d.batch.chunk_table([(0, 60_000), (60_000, 120_000)]))
    assert rec.size > 8


def test_dense_candidates(ctx):
    """10 % substitutions and no window / identity gate: nearly every position of a tile is a site (the (ref, alt)
    masks leave shared memory), every read has thousands of ops (op arrays leave shared memory), and the first guess
    of the site count is too small"""
    d = synth.generate(150_000, seed=5, sub_err_rate=0.1)
    a = dict(gtmodel.DEFAULT_CALL_ARGS, max_mismatch_count=100000, min_sequence_identity=0.0)
    p = gtmodel.make_params(**a)
    rec, log = _same_as_oracle(ctx, p, d.batch, d.batch.chunk_table([(0, 150_000)]))
    assert rec.size > 100_000
    _same_as_oracle(ctx, p, d.batch.without_seq(), d.batch.chunk_table([(0, 75_000), (75_000, 150_000)]), full=d.batch)


def test_reads_that_fail_the_qv_gate_emit_no_candidates(ctx):
    """the QV gate (the read's resident quality sum) decides before any candidate of the read is emitted; a site none
    of whose supporting reads passes it must vanish (records, counters, num_ccs)"""
    d = synth.generate(200_000, seed=11)
    b = d.batch
    for r in range(0, b.n_reads, 3):  # every third read: qualities 20 everywhere (mean < min_qv = 30)
        o = int(b.bq_off[r])
        b.bq[o:o + int(b.qlen[r])] = 20
    p = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
    chunks = b.chunk_table(cases.chunkloci(0, 200_000))
    rec, log = _same_as_oracle(ctx, p, b, chunks)
    full = gtmodel.make_params(**dict(gtmodel.DEFAULT_CALL_ARGS, min_qv=0))
    rec0, log0 = _same_as_oracle(ctx, full, b, chunks)
    assert log[0] < log0[0] and log[1] < log0[1]  # fewer reads counted, fewer sites evaluated


def test_empty_tail_chunks_and_negative_spans(ctx):
    d = synth.generate(60_000, seed=5)
    p = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
    chunks = d.batch.chunk_table([(0, 30_000), (30_000, 60_000), (59_000, 58_000), (10_000, 10_000)])
    _same_as_oracle(ctx, p, d.batch, chunks)
