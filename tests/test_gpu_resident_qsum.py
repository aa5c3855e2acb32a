"""The QV gate reads the per-read quality sum the resident batch carries (DevBatch.bq_total), written when the batch
becomes resident: k_bq_sum after a plain upload or a device BAM decode, k_bq_expand after a compact upload.  Reads
whose mean quality is exactly min_qv pass the gate and reads one quality point short of it fail, on every way a batch
becomes resident; two batches one after the other on one context catch a sum left over from the first.  Records and
all 15 counters against the oracle.  GPU."""
import numpy as np
import pytest

import cases
import parity
from himut_b200 import abi, bamdec, gtmodel, synth
from oracle import oracle

pytestmark = pytest.mark.gpu
N = 200_000
PARAMS = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
MIN_QV = gtmodel.DEFAULT_CALL_ARGS["min_qv"]


def _with_bq(batch, bq):
    kw = {name: getattr(batch, name) for name, _ in abi.ReadBatch._FIELDS}
    kw["bq"] = bq
    return abi.ReadBatch(**kw)


def _boundary_batch(batch):
    """every third read: mean quality exactly min_qv (passes); the read after it: the same less one point on its
    first base (its integer sum is one below min_qv * qlen: fails); the rest as generated"""
    bq = batch.bq.copy()
    for r in range(0, batch.n_reads - 1, 3):
        for k, short in ((r, 0), (r + 1, 1)):
            o, n = int(batch.bq_off[k]), int(batch.qlen[k])
            bq[o:o + n] = MIN_QV
            bq[o] -= short
    return _with_bq(batch, bq)


def _lowered(batch):
    """the same reads with every third read's qualities below the gate"""
    bq = batch.bq.copy()
    for r in range(0, batch.n_reads, 3):
        o, n = int(batch.bq_off[r]), int(batch.qlen[r])
        bq[o:o + n] = MIN_QV - 5
    return _with_bq(batch, bq)


def _check(rec, log, batch, chunks):
    o_rec, o_log = oracle.call_chunks(PARAMS, batch, chunks)
    ok, why = parity.records_equal(rec, o_rec)
    assert ok, why
    assert list(log) == list(o_log)
    return list(log)


def _plain(ctx, batch, chunks):
    ctx.upload(batch.without_seq())
    rec, log = ctx.call_chunks(chunks)
    assert ctx.last_call_path() == 2
    return _check(rec, log, batch, chunks)


def _compact(ctx, batch, chunks):
    """upload_compact without waiting, the call submitted straight behind it (as the worker does)"""
    b = batch.without_seq()
    cq = bamdec.compact_bq(b)
    ctx.upload_compact(b, cq, wait=False)
    ctx.call_chunks_submit(chunks)
    rec, log = ctx.call_chunks_collect(view=False)
    ctx.upload_wait()
    assert ctx.last_call_path() == 2
    return _check(rec, log, batch, chunks)


@pytest.fixture(scope="module")
def data():
    d = synth.generate(N, seed=23)
    return _boundary_batch(d.batch), d.batch.chunk_table(cases.chunkloci(0, N))


def _gate_matters(ctx, batch, chunks, log):
    """the gate decided something: without it more reads count"""
    ctx.set_params(gtmodel.make_params(**dict(gtmodel.DEFAULT_CALL_ARGS, min_qv=0)))
    try:
        ctx.upload(batch.without_seq())
        _, log0 = ctx.call_chunks(chunks)
    finally:
        ctx.set_params(PARAMS)
    assert log[0] < log0[0]


def test_boundary_plain_upload(ctx, data):
    batch, chunks = data
    ctx.set_params(PARAMS)
    ctx.set_site_sets()
    log = _plain(ctx, batch, chunks)
    _gate_matters(ctx, batch, chunks, log)


def test_boundary_compact_upload_not_waited_for(ctx, data):
    batch, chunks = data
    ctx.set_params(PARAMS)
    ctx.set_site_sets()
    assert _compact(ctx, batch, chunks) == _plain(ctx, batch, chunks)


def test_boundary_device_decode(ctx, data, tmp_path):
    batch, chunks = data
    ctx.set_params(PARAMS)
    ctx.set_site_sets()
    path = str(tmp_path / "q.bam")
    bamdec.write_batch_bam(path, "chr1", N, batch)
    nb = bamdec.NativeBam(path, threads=2)
    try:
        host = nb.read_batch("chr1", 0, N, seq=True)
        region = ctx.decode_region(nb, "chr1", 0, N)
    finally:
        nb.close()
    assert region.n_reads == host.n_reads
    hchunks = host.chunk_table(cases.chunkloci(0, N))
    rec, log = ctx.call_chunks(hchunks)
    assert ctx.last_call_path() == 2
    assert _check(rec, log, host, hchunks) == _plain(ctx, host, hchunks)


@pytest.mark.parametrize("order", [("plain", "compact"), ("compact", "plain")])
def test_second_batch_on_the_same_context(ctx, data, order):
    batch, chunks = data
    ctx.set_params(PARAMS)
    ctx.set_site_sets()
    up = {"plain": _plain, "compact": _compact}
    first = up[order[0]](ctx, batch, chunks)
    second = up[order[1]](ctx, _lowered(batch), chunks)
    assert second[0] < first[0]
