"""Device BAM decoder on records with neither cs:Z nor MD:Z (CIGAR + the resident reference, HM_DECODE_REF): the
resident batch against the host decoder byte for byte, with and without the base stream, the rejections of the
reference path with the host's words, and `call`, normcounts and the phase edges decoded on the device from eqx / m
BAMs against the same batches written with cs.  GPU."""
import json
import os

import numpy as np
import pytest

import cases
import parity
import test_bamdec as tb
import test_edges as te
import test_gpu_bamdecode as tg
import test_gpu_bamdecode_seq as ts
import test_gpu_md_ops as tgm
import test_ref_ops as tr
from himut_b200 import abi, bamdec, bamio, caller, gtmodel, lib, normcounts, pack, phaselib, synth, worker

pytestmark = pytest.mark.gpu

KERNELS = tg.DECODE_KERNELS | {"k_bam_ref_count"}


def _same_as_host(ctx, nb, ref, s, e, seq):
    """the device batch of [s, e) = the host decoder's, the reference set on both"""
    nb.set_reference("chr1", ref)
    want = nb.read_batch("chr1", s, e, seq=seq)
    r = ctx.decode_region(nb, "chr1", s, e, seq=seq, ref=ref)
    assert r.n_reads == 0 or KERNELS <= {k for k, _ in ctx.last_decode_times}
    got = ctx.read_back(seq=seq)
    for name in (ts.FIELDS if seq else ts.FIELDS[:-2]):
        x, y = getattr(got, name), getattr(want, name)
        assert x.shape == y.shape and np.array_equal(x, y), (name, s, e, seq)
    return got


@pytest.mark.parametrize("writer", ["python", "native"])
@pytest.mark.parametrize("tags", ["eqx", "m"])
def test_device_ref_batch_equals_host_batch(ctx, tmp_path, writer, tags):
    n = 300_000
    d = synth.generate(n, seed=11)
    path = str(tmp_path / "t.bam")
    (bamio.write_batch_bam if writer == "python" else bamdec.write_batch_bam)(path, "chr1", n, d.batch, tags=tags)
    nb = bamdec.NativeBam(path, threads=4)
    for s, e in tgm.WINDOWS:
        for seq in (False, True):
            _same_as_host(ctx, nb, d.ref, s, e, seq)
    nb.close()


def test_device_adversarial_and_mixed_ref(ctx, tmp_path):
    """dense events, N reference letters, clips, secondary records; cs, MD and tag-less records alternating"""
    for seed in (1, 2, 5):
        batch, ref = cases.adversarial_batch(seed, contig_len=6000, n_reads=300, max_len=2000)
        path = str(tmp_path / ("a%d.bam" % seed))
        bamdec.write_batch_bam(path, "chr1", 6000, batch, tags="m" if seed != 2 else "eqx")
        nb = bamdec.NativeBam(path, threads=2)
        for s, e in ((0, 6000), (1000, 1001), (2500, 4000)):
            for seq in (False, True):
                _same_as_host(ctx, nb, ref.encode(), s, e, seq)
        nb.close()
    n = 100_000
    d = synth.generate(n, seed=7)
    paths = tr._paths(tmp_path, n, d.batch, forms=("cs", "md", "eqx"), writer="python")
    forms = [list(bamio.BamReader(paths[t]).fetch("chr1")) for t in ("cs", "md", "eqx")]
    p_mix = str(tmp_path / "mix.bam")
    w = bamio.BamWriter(p_mix, [("chr1", n)])
    for i, r in enumerate(zip(*forms)):
        r = r[i % 3]
        w.add(r.ref_id, r.reference_start, r.query_name, r.flag, r.mapping_quality, r.cigar, r.query_sequence, bytes(r.qual),
              [(t, "A" if t == "tp" else "Z", v) for t, v in r.tags.items()])
    w.close()
    nb = bamdec.NativeBam(p_mix, threads=2)
    got = _same_as_host(ctx, nb, d.ref, 0, n, True)
    nb.close()
    want = bamdec.NativeBam(paths["cs"], threads=2).read_batch("chr1", 0, n, seq=True)
    for name in ts.FIELDS:
        assert np.array_equal(getattr(got, name), getattr(want, name)), name


def _device_error(ctx, path, ref):
    nb = bamdec.NativeBam(path, threads=1)
    try:
        with pytest.raises(pack.BatchFormatError) as ex:
            ctx.decode_region(nb, "chr1", 0, 1000, ref=ref)
        return str(ex.value)
    finally:
        nb.close()


@pytest.mark.parametrize("bad, key, arg", tr.REF_BAD)
def test_device_ref_rejections_match_the_host(ctx, tmp_path, bad, key, arg):
    path = str(tmp_path / "b.bam")
    tb._write(path, [tr._ref_rec(qname="refrec", **bad)])
    want = (pack.REF_ERR.get(key) or pack.MD_ERR[key]) % ("refrec", arg)
    assert _device_error(ctx, path, tr.TB_REF) == want
    nb = bamdec.NativeBam(path, threads=1)
    nb.set_reference("chr1", tr.TB_REF)
    with pytest.raises(pack.BatchFormatError) as ex:
        ctx.decode_region(nb, "chr1", 0, 1000, seq=True, ref=True)
    assert str(ex.value) == want
    nb.close()


def test_device_ref_needs_a_resident_reference_and_the_bit(ctx, tmp_path):
    path = str(tmp_path / "b.bam")
    tb._write(path, [tr._ref_rec(qname="bare")])
    # without the bit a tag-less record is still "no cs:Z tag", reference resident or not
    ctx.set_reference(tr.TB_REF)
    assert tg._device_error(ctx, path).startswith("bare has no cs:Z tag")
    nb = bamdec.NativeBam(path, threads=1)
    ctx.ref_tricounts(tr.TB_REF)  # replaces the resident reference: none is left
    plan = nb.plan("chr1", 0, 1000)
    import ctypes as C
    n = C.c_uint64(0)
    rc = ctx.lib.hm_decode_bam_begin_opts(ctx.h, C.byref(plan), 0, 0, 1000, abi.HM_DECODE_REF, C.byref(n))
    assert rc == abi.HM_ERR_STATE
    assert ctx.decode_region(nb, "chr1", 0, 1000, ref=tr.TB_REF).n_reads == 1
    nb.close()


def test_decode_region_refuses_a_reference_of_another_length_or_type(ctx, tmp_path):
    """a resident sequence that is not the contig's (its length is not @SQ LN) never reaches the decoder"""
    path = str(tmp_path / "b.bam")
    tb._write(path, [tr._ref_rec(qname="r")])
    nb = bamdec.NativeBam(path, threads=1)
    with pytest.raises(ValueError, match="has 999 bases, contig chr1 of the BAM 1000"):
        ctx.decode_region(nb, "chr1", 0, 1000, ref=tr.TB_REF[:999])
    with pytest.raises(ValueError, match="has 999 bases"):
        ctx.decode_region(nb, "chr1", 0, 1000, ref=True)
    with pytest.raises(TypeError):
        ctx.decode_region(nb, "chr1", 0, 1000, ref=tr.TB_REF.decode())
    assert ctx.decode_region(nb, "chr1", 0, 1000, ref=tr.TB_REF).n_reads == 1
    nb.close()


def _tagless_bams(monkeypatch, tags):
    tgm._md_bams(monkeypatch, tags)


def test_call_worker_device_decode_m_config0(tmp_path, monkeypatch):
    """BASELINE configs[0] (1 Mb) written as M CIGARs without a tag: the drop-in get_somatic_substitutions, its FASTA
    from HIMUT_B200_REF, fills the golden rows"""
    c = cases.build_case("call_config0_1mb")
    fx = parity.load_golden("call_config0_1mb")
    fa = str(tmp_path / "ref.fa")
    tr.write_fasta(fa, [(cases.CHROM, c["ref"], "")])
    monkeypatch.setenv("HIMUT_B200_REF", fa)
    _tagless_bams(monkeypatch, "m")
    rows, log = tg._run_call_device(c, tmp_path, monkeypatch)
    gold = parity.golden_rows(fx)
    assert parity.rows_equal(rows, gold), parity.first_diff(rows, gold)
    assert log == fx["expected"]["log"]


def test_normcounts_worker_device_decode_eqx_config0(tmp_path, monkeypatch):
    c = cases.build_case("norm_config0_1mb")
    want = ts._run_norm(c, tmp_path, monkeypatch, "device")
    _tagless_bams(monkeypatch, "eqx")
    assert ts._run_norm(c, tmp_path, monkeypatch, "device") == want


@pytest.mark.parametrize("name", ["plain", "bq0_counts_deletions"])
def test_phase_edges_device_decode_m(tmp_path, monkeypatch, name):
    batch, hetsnp_lst, h2i, n, min_bq, min_mapq = te.mk.inputs(name)
    ref = _agreeing_reference(batch, n)
    path = str(tmp_path / "e.bam")
    bamdec.write_batch_bam(path, "chr1", n, batch, tags="m")
    fa = str(tmp_path / "ref.fa")
    tr.write_fasta(fa, [("chr1", ref, "")])
    monkeypatch.setenv("HIMUT_B200_REF", fa)
    real = phaselib.edge_table
    monkeypatch.setattr(phaselib, "edge_table", lambda *a, **k: real(*a, **dict(k, decode="device")))
    edge_lst, e2c = phaselib.get_edges("chr1", path, min_bq, min_mapq, [h[0] for h in hetsnp_lst], hetsnp_lst, h2i)
    got = [[int(i), int(j)] + [int(v) for v in e2c[(i, j)]] for (i, j) in edge_lst]
    assert got == json.load(open(os.path.join(cases.GOLDEN_DIR, "edges.json")))["expected"][name]


def _agreeing_reference(batch, n):
    """a reference the batch agrees with: the read base under each MATCH, each SUB's reference base, N elsewhere"""
    ref = bytearray(b"N" * n)
    for r in range(batch.n_reads):
        so, oo, ql = int(batch.seq_off[r]), int(batch.op_off[r]), int(batch.qlen[r])
        codes = ((batch.seq[so:so + (ql + 3) // 4][:, None] >> np.array([0, 2, 4, 6], np.uint8)) & 3).reshape(-1)[:ql]
        t, q = int(batch.tstart[r]), int(batch.qstart[r])
        for w in batch.ops[oo:oo + int(batch.n_ops[r])]:
            kind, val = int(w) & 3, int(w) >> 2
            if kind == abi.OP_MATCH:
                ref[t:t + val] = bytes(b"ATGC"[c] for c in codes[q:q + val]); t += val; q += val
            elif kind == abi.OP_SUB:
                ref[t] = b"ATGCN"[min(val & 7, 4)]; t += 1; q += 1
            elif kind == abi.OP_INS:
                q += val
            else:
                t += val
    return bytes(ref)


def test_one_16mb_group_eqx_and_m_equal_cs(tmp_path):
    """one full decode group (worker.GROUP_SPAN) of a 30x contig: call, normcounts and the phase edges decoded on the
    device from the eqx and m BAMs give what they give from the cs BAM (each on a fresh context)"""
    n = worker.GROUP_SPAN
    d = synth.generate(n, seed=5, copy=False)
    ref = bytes(d.ref)
    paths = {}
    for tags in ("cs", "eqx", "m"):
        paths[tags] = str(tmp_path / ("%s.bam" % tags))
        bamdec.write_batch_bam(paths[tags], "chr1", n, d.batch, tags=tags)
    hpos = np.asarray(d.germ["pos"], np.int32)[:20_000]
    href = np.asarray(d.germ["ref"], np.uint8)[:20_000]
    del d
    loci = [("chr1", s, e) for s, e in cases.chunkloci(0, n)]
    out = {}
    for tags, path in paths.items():
        res = []
        for run in ("call", "norm", "edges"):
            with lib.Context(0) as ctx:
                ctx.set_params(gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS))
                ctx.set_site_sets()
                if run == "call":
                    res.append(caller.call_region(ctx, path, "chr1", loci, None, None, decode="device", refseq=ref))
                elif run == "norm":
                    res.append(normcounts.normcounts_region(ctx, path, "chr1", ref, loci, None, decode="device"))
                else:
                    res.append(phaselib.edge_table(ctx, path, "chr1", hpos, href, 10, 20, decode="device", refseq=ref))
        out[tags] = res
    tgm._deep_equal(out["cs"], out["eqx"])
    tgm._deep_equal(out["cs"], out["m"])
