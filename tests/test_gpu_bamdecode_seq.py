"""Device BAM decoder with the 2-bit base stream (hm_decode_bam_begin_opts(HM_DECODE_SEQ)): the resident batch against
the host decoder's batch with seq byte for byte, the host decoder's rejections, no state carried between decodes, and
the normcounts worker and the phase edges on the device decode path against the reference's outputs.  GPU."""
import json
import os
import random

import numpy as np
import pytest

import cases
import parity
import test_bamdec as tb
import test_edges as te
import test_gpu_bamdecode as tg
import test_gpu_worker as tw
from himut_b200 import abi, bamdec, bamio, gtmodel, lib, normcounts, pack, phaselib, synth, worker

pytestmark = pytest.mark.gpu

FIELDS = ("tstart", "tend", "qstart", "qlen", "mapq", "qname_id", "bq_off", "op_off", "n_ops", "bq", "ops", "seq_off", "seq")


def _same_as_host(ctx, nb, chrom, s, e):
    want = nb.read_batch(chrom, s, e, seq=True)
    r = ctx.decode_region(nb, chrom, s, e, seq=True)
    ran = {k for k, _ in ctx.last_decode_times}
    assert r.n_reads == 0 or tg.DECODE_KERNELS <= ran  # a contig without records plans no block: nothing runs
    got = ctx.read_back(seq=True)
    assert got.n_reads == r.n_reads and np.array_equal(got.tstart, r.tstart) and np.array_equal(got.tend, r.tend)
    for name in FIELDS:
        x, y = getattr(got, name), getattr(want, name)
        assert x.shape == y.shape and np.array_equal(x, y), (name, chrom, s, e)
    return got


@pytest.mark.parametrize("writer", ["python", "native"])
@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_device_seq_batch_equals_host_batch(ctx, tmp_path, writer, level):
    n = 300_000
    d = synth.generate(n, seed=11)
    path = str(tmp_path / "t.bam")
    tg._write_level(path, [("chr1", n, d.batch)], writer, level)
    nb = bamdec.NativeBam(path, threads=4)
    for s, e in [(0, n), (1, 200_000), (200_000, 299_998), (123_456, 123_457), (299_990, n), (0, 1), (n + 5, n + 50)]:
        _same_as_host(ctx, nb, "chr1", s, e)
    nb.close()


def test_device_seq_clips_iupac_secondary_supplementary_longform(ctx, tmp_path):
    path = str(tmp_path / "m.bam")
    tb._write(path, [
        tb._rec(pos=10, cigar=((4, 2), (0, 6), (4, 1)), seq="NNACGTACN", cs=":6", qname="clip"),
        tb._rec(pos=11, cigar=((4, 5), (0, 6), (4, 4)), seq="RYKM=ACGTACSWBD", cs=":6", qname="iupac"),
        tb._rec(pos=12, flag=0x100, qname="secondary", cs=None),
        tb._rec(pos=14, flag=0x800, qname="supp", cs=":3*ag:2+tt-ca:0", cigar=((0, 6), (1, 2), (2, 2)), seq="ACGGACTT"),
        tb._rec(pos=16, cigar=((5, 3), (0, 8), (5, 2)), qname="hardclip"),
        tb._rec(pos=20, cs="=ACGT*ct=CGT", seq="ACGTTCGT", qname="longform"),
        tb._rec(pos=5, ref_id=1, qname="other"),
    ])
    nb = bamdec.NativeBam(path, threads=1)
    for chrom in ("chr1", "chr2"):
        for s, e in [(0, 1000), (15, 16), (0, 11), (27, 40)]:
            _same_as_host(ctx, nb, chrom, s, e)
    assert _same_as_host(ctx, nb, "chr1", 0, 1000).n_reads == 5
    nb.close()


def test_device_seq_at_every_read_length(ctx, tmp_path):
    """lengths 1-40 cross the nibble, 4-base, 16-byte and lane boundaries of the packing; 500-1100 make a lane pack
    more than one word; N / IUPAC / '=' letters in the soft clips are stored as 0"""
    rnd = random.Random(9)
    recs = []
    for k, n in enumerate(list(range(1, 41)) + [63, 64, 65, 127, 128, 129, 511, 512, 513, 1100]):
        lead, trail = rnd.randrange(0, 4), rnd.randrange(0, 4)
        m = max(1, n - lead - trail)
        lead = min(lead, n - m)
        trail = n - m - lead
        clip = lambda j: "".join(rnd.choice("ACGTNRY=") for _ in range(j))
        body = "".join(rnd.choice("ACGT") for _ in range(m))
        cigar = ([(4, lead)] if lead else []) + [(0, m)] + ([(4, trail)] if trail else [])
        recs.append(tb._rec(pos=10 + k, cigar=cigar, seq=clip(lead) + body + clip(trail), cs=":%d" % m, qname="r%d" % n))
    path = str(tmp_path / "len.bam")
    tb._write(path, recs, reflen=5000)
    nb = bamdec.NativeBam(path, threads=2)
    got = _same_as_host(ctx, nb, "chr1", 0, 5000)
    assert got.n_reads == len(recs) and sorted(got.qlen.tolist()) == sorted(len(r["seq"]) for r in recs)
    nb.close()


def test_device_seq_multi_contig_and_without_index(ctx, tmp_path):
    a, b = synth.generate(60_000, seed=22), synth.generate(40_000, seed=23)
    path = str(tmp_path / "m.bam")
    bamio.write_batches_bam(path, [("chr1", 60_000, a.batch), ("chr2", 40_000, b.batch)])
    nb = bamdec.NativeBam(path, threads=2)
    for chrom, n in (("chr1", 60_000), ("chr2", 40_000)):
        for s, e in ((0, n), (n // 3, n // 2), (n - 1, n)):
            _same_as_host(ctx, nb, chrom, s, e)
    nb.close()
    os.remove(path + ".bai")
    nb = bamdec.NativeBam(path, threads=2)
    assert not nb.has_index
    for chrom, n in (("chr1", 60_000), ("chr2", 40_000)):
        _same_as_host(ctx, nb, chrom, n // 4, n // 2)
    nb.close()


def test_device_seq_empty_region(ctx, tmp_path):
    """no reads: 16 zero base bytes and 16 zero quality bytes, as the host decoder leaves its empty batch"""
    path = str(tmp_path / "m.bam")
    tb._write(path, [tb._rec(pos=10, qname="a"), tb._rec(pos=500, qname="b")])
    nb = bamdec.NativeBam(path, threads=1)
    for chrom, s, e in (("chr1", 100, 400), ("chr2", 0, 1000), ("chr1", 990, 1000)):
        got = _same_as_host(ctx, nb, chrom, s, e)
        assert got.n_reads == 0 and got.seq.tolist() == [0] * 16 and got.bq.tolist() == [0] * 16
    nb.close()


@pytest.fixture(scope="module")
def contig_64mb(tmp_path_factory):
    """the contig of tools/worker_trace.py (64 Mb, 30x, seed 5) -> (path, length, reference)"""
    n = 64_000_000
    d = synth.generate(n, seed=5, copy=False)
    path = str(tmp_path_factory.mktemp("c64") / "c.bam")
    bamdec.write_batch_bam(path, "chr1", n, d.batch)
    ref = bytes(d.ref)
    del d
    return path, n, ref


def test_device_seq_batch_of_the_64mb_contig(ctx, contig_64mb):
    path, n, _ref = contig_64mb
    nb = bamdec.NativeBam(path)
    for s, e in [(0, n)] + [(g, g + 16_000_000) for g in range(0, n, 16_000_000)]:
        _same_as_host(ctx, nb, "chr1", s, e)
    nb.close()


def _device_error(ctx, path, s=0, e=1000):
    nb = bamdec.NativeBam(path, threads=1)
    try:
        with pytest.raises(pack.BatchFormatError) as ex:
            ctx.decode_region(nb, "chr1", s, e, seq=True)
        return str(ex.value)
    finally:
        nb.close()


def _host_error(path, s=0, e=1000):
    nb = bamdec.NativeBam(path, threads=1)
    try:
        with pytest.raises(pack.BatchFormatError) as ex:
            nb.read_batch("chr1", s, e, seq=True)
        return str(ex.value)
    finally:
        nb.close()


@pytest.mark.parametrize("bad", [
    dict(cs=None), dict(seq="ACNTACGT"), dict(cs=":2*an:5"), dict(cs=":9"), dict(cs=":7"), dict(cs=":4~gt12ag:4"),
    dict(qual=b"\xff" * 8),
])
def test_device_seq_rejections_match_the_host(ctx, tmp_path, bad):
    path = str(tmp_path / "b.bam")
    tb._write(path, [tb._rec(**bad)])
    assert _device_error(ctx, path) == _host_error(path)


def test_device_seq_reports_the_record_the_host_reports(ctx, tmp_path):
    path = str(tmp_path / "two.bam")
    tb._write(path, [tb._rec(pos=10, cs=":7", qname="badcs"), tb._rec(pos=20, cs=None, qname="nocs")])
    msg = _host_error(path)
    assert msg.startswith("nocs has no cs:Z tag")
    assert _device_error(ctx, path) == msg


def test_no_state_carried_between_decodes(tmp_path):
    """on one context: a decode without seq after one with it leaves a batch without a base stream (normcounts refuses
    it as it refuses the host decoder's no-seq batch); a decode with seq after one without leaves the whole batch"""
    d = synth.generate(100_000, seed=41)
    path = str(tmp_path / "t.bam")
    bamdec.write_batch_bam(path, "chr1", 100_000, d.batch)
    nb = bamdec.NativeBam(path, threads=2)
    with lib.Context(0) as c:
        c.set_params(gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS))
        c.set_site_sets()
        for first, second in ((True, False), (False, True), (True, True)):
            c.decode_region(nb, "chr1", 0, 100_000, seq=first)
            region = c.decode_region(nb, "chr1", 20_000, 80_000, seq=second)
            table = region.chunk_table([(20_000, 80_000)])
            got = c.read_back(seq=True)
            if second:
                want = nb.read_batch("chr1", 20_000, 80_000, seq=True)
                for name in FIELDS:
                    assert np.array_equal(getattr(got, name), getattr(want, name)), (first, second, name)
                c.normcounts_chunks(d.ref, table)
            else:
                assert got.seq.size == 0 and got.seq_off.size == 0
                with pytest.raises(lib.HimutError) as ex:
                    c.normcounts_chunks(d.ref, table)
                assert ex.value.code == abi.HM_ERR_STATE
    nb.close()


def _spy_decodes(monkeypatch):
    seen = []
    orig = lib.Context.decode_region

    def spy(self, *a, **k):
        r = orig(self, *a, **k)
        seen.append(({n for n, _ in self.last_decode_times}, bool(k.get("seq"))))
        return r

    monkeypatch.setattr(lib.Context, "decode_region", spy)
    return seen


def _run_norm(c, tmp_path, monkeypatch, decode):
    real = normcounts.normcounts_region
    monkeypatch.setattr(normcounts, "normcounts_region", lambda *a, **k: real(*a, **dict(k, decode=decode)))
    a = c["args"]
    bam, common, pon = tw._inputs(c, tmp_path)
    hbit, hpos, hetsnp = cases.phase_dicts(c)
    ccs, rt, log = {}, {}, {}
    ties = normcounts.get_callable_tricounts(
        cases.CHROM, c["ref"], bam, common, pon, [(cases.CHROM, s, e2) for s, e2 in c["chunks"]], hbit, hpos, hetsnp,
        a["min_qv"], a["min_mapq"], a["min_trim"], a["qlen_lower_limit"], a["qlen_upper_limit"],
        a["min_sequence_identity"], a["min_gq"], a["min_bq"], a["mismatch_window"], a["max_mismatch_count"],
        a["min_ref_count"], a["min_alt_count"], a["min_hap_count"], float(a["md_threshold"]), 1e-6,
        a["germline_snv_prior"], 1e-4, bool(a.get("phase")), bool(a.get("non_human_sample")), ccs, rt, log)
    monkeypatch.setattr(normcounts, "normcounts_region", real)
    return ccs[cases.CHROM], rt[cases.CHROM], log[cases.CHROM], ties


@pytest.mark.parametrize("name", ["norm_basic", "norm_sets", "norm_phase", "norm_adversarial", "norm_config3_phase_sets",
                                  "norm_config0_1mb"])
def test_normcounts_worker_device_decode_matches_reference(name, tmp_path, monkeypatch):
    """the worker with decode="device" equals the worker with decode="host", and the reference's outputs wherever the
    reference's own result does not depend on its hash seed (no alt ties)"""
    if name == "norm_adversarial":
        monkeypatch.setattr(worker, "GROUP_SPAN", 1200)
    c = cases.build_case(name)
    e = parity.load_golden(name)["expected"]
    seen = _spy_decodes(monkeypatch)
    got = _run_norm(c, tmp_path, monkeypatch, "device")
    assert seen and all(s for _, s in seen) and any(tg.DECODE_KERNELS <= k for k, _ in seen)
    n_dev = len(seen)
    assert _run_norm(c, tmp_path, monkeypatch, "host") == got
    assert len(seen) == n_dev
    ccs, rt, log, ties = got
    if not ties:
        for tri in normcounts.TRI_LST:
            assert ccs[tri] == e["ccs_tri2count"].get(tri, 0), tri
            assert rt[tri] == e["ref_tri2count"].get(tri, 0), tri
        assert log == e["log"]


@pytest.mark.parametrize("name", ["plain", "bq0_counts_deletions"])
@pytest.mark.parametrize("span", [37_000, 10_000_000])
def test_phase_edges_device_decode_matches_reference(tmp_path, monkeypatch, name, span):
    batch, hetsnp_lst, h2i, n, min_bq, min_mapq = te.mk.inputs(name)
    path = str(tmp_path / "e.bam")
    bamdec.write_batch_bam(path, "chr1", n, batch)
    monkeypatch.setattr(worker, "GROUP_SPAN", span)
    seen = _spy_decodes(monkeypatch)
    real = phaselib.edge_table
    monkeypatch.setattr(phaselib, "edge_table", lambda *a, **k: real(*a, **dict(k, decode="device")))
    edge_lst, e2c = phaselib.get_edges("chr1", path, min_bq, min_mapq, [h[0] for h in hetsnp_lst], hetsnp_lst, h2i)
    assert seen and not any(s for _, s in seen) and any(tg.DECODE_KERNELS <= k for k, _ in seen)
    got = [[int(i), int(j)] + [int(v) for v in e2c[(i, j)]] for (i, j) in edge_lst]
    assert got == json.load(open(os.path.join(cases.GOLDEN_DIR, "edges.json")))["expected"][name]
    assert all(isinstance(v, np.ndarray) and v.dtype == np.float64 for v in e2c.values())


def test_normcounts_worker_64mb_device_equals_host(ctx, contig_64mb, monkeypatch):
    path, n, ref = contig_64mb
    ctx.set_params(gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS))
    ctx.set_site_sets()
    loci = [("chr1", s, e) for s, e in cases.chunkloci(0, n)]
    seen = _spy_decodes(monkeypatch)
    host = normcounts.normcounts_region(ctx, path, "chr1", ref, loci, None, decode="host")
    assert not seen
    dev = normcounts.normcounts_region(ctx, path, "chr1", ref, loci, None, decode="device")
    assert len(seen) == len(worker.group_chunks(loci)) and all(tg.DECODE_KERNELS <= k and s for k, s in seen)
    for x, y in zip(host, dev):  # tri counts, log, alt ties, distinct names
        assert np.array_equal(x, y)
    assert int(host[2][13]) > 32 * 20_000_000
