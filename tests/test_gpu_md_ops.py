"""Device BAM decoder on records without cs:Z (CIGAR + MD:Z): the resident batch against the host decoder byte for byte,
with and without the base stream, the rejections of the MD path with the host's words, and `call`, normcounts and
the phase edges decoded on the device from MD BAMs against the same batches written with cs.  GPU."""
import json
import os

import numpy as np
import numpy.lib.recfunctions as rfn
import pytest

import cases
import parity
import test_bamdec as tb
import test_gpu_bamdecode as tg
import test_gpu_bamdecode_seq as ts
import test_edges as te
import test_md_ops as tm
from himut_b200 import bamdec, bamio, caller, gtmodel, lib, normcounts, phaselib, synth, worker

pytestmark = pytest.mark.gpu

WINDOWS = [(0, 300_000), (1, 200_000), (200_000, 299_998), (123_456, 123_457), (299_990, 300_000), (0, 1), (300_005, 300_050)]


@pytest.mark.parametrize("writer", ["python", "native"])
@pytest.mark.parametrize("tags", ["md", "md_eqx"])
def test_device_md_batch_equals_host_batch(ctx, tmp_path, writer, tags):
    n = 300_000
    d = synth.generate(n, seed=11)
    path = str(tmp_path / "t.bam")
    (bamio.write_batch_bam if writer == "python" else bamdec.write_batch_bam)(path, "chr1", n, d.batch, tags=tags)
    nb = bamdec.NativeBam(path, threads=4)
    for s, e in WINDOWS:
        tg._same_as_host(ctx, nb, "chr1", s, e)
        ts._same_as_host(ctx, nb, "chr1", s, e)
    nb.close()


def test_device_adversarial_and_mixed_md(ctx, tmp_path):
    """dense events, N reference letters, clips, secondary records; cs and MD records alternating in one file"""
    for seed in (1, 2, 5):
        batch, _ref = cases.adversarial_batch(seed, contig_len=6000, n_reads=300, max_len=2000)
        path = str(tmp_path / ("a%d.bam" % seed))
        bamdec.write_batch_bam(path, "chr1", 6000, batch, tags="md" if seed != 2 else "md_eqx")
        nb = bamdec.NativeBam(path, threads=2)
        for s, e in ((0, 6000), (1000, 1001), (2500, 4000)):
            tg._same_as_host(ctx, nb, "chr1", s, e)
            ts._same_as_host(ctx, nb, "chr1", s, e)
        nb.close()
    n = 100_000
    d = synth.generate(n, seed=7)
    p_cs, p_md, p_mix = (str(tmp_path / x) for x in ("cs.bam", "md.bam", "mix.bam"))
    bamio.write_batch_bam(p_cs, "chr1", n, d.batch)
    bamio.write_batch_bam(p_md, "chr1", n, d.batch, tags="md")
    w = bamio.BamWriter(p_mix, [("chr1", n)])
    for i, (x, y) in enumerate(zip(bamio.BamReader(p_cs).fetch("chr1"), bamio.BamReader(p_md).fetch("chr1"))):
        r = x if i % 3 else y
        w.add(r.ref_id, r.reference_start, r.query_name, r.flag, r.mapping_quality, r.cigar, r.query_sequence, bytes(r.qual),
              [(t, "A" if t == "tp" else "Z", v) for t, v in r.tags.items()])
    w.close()
    nb = bamdec.NativeBam(p_mix, threads=2)
    got = ts._same_as_host(ctx, nb, "chr1", 0, n)
    nb.close()
    nb = bamdec.NativeBam(p_cs, threads=2)
    want = nb.read_batch("chr1", 0, n, seq=True)
    nb.close()
    for name in ts.FIELDS:
        assert np.array_equal(getattr(got, name), getattr(want, name)), name


@pytest.mark.parametrize("bad, key, arg", tm.MD_BAD + [(dict(cs=None), None, None)])
def test_device_md_rejections_match_the_host(ctx, tmp_path, bad, key, arg):
    path = str(tmp_path / "b.bam")
    rec = tm._md_rec(qname="mdrec", **bad) if key else tb._rec(qname="mdrec", **bad)
    tb._write(path, [rec])
    want = tg._host_error(path)
    if key:
        assert want == tm.pack.MD_ERR[key] % ("mdrec", arg)
    else:
        assert want.startswith("mdrec has no cs:Z tag")
    assert tg._device_error(ctx, path) == want
    assert ts._device_error(ctx, path) == ts._host_error(path) == want


def _md_bams(monkeypatch, tags="md"):
    """the tests' BAM writers write MD instead of cs from here on"""
    for mod, real in ((bamio, bamio.write_batch_bam), (bamdec, bamdec.write_batch_bam)):
        monkeypatch.setattr(mod, "write_batch_bam", lambda *a, _real=real, **k: _real(*a, **dict(k, tags=tags)))


def test_call_worker_device_decode_md_config0(tmp_path, monkeypatch):
    """BASELINE configs[0] (1 Mb) written as MD: the drop-in get_somatic_substitutions fills the golden rows"""
    c = cases.build_case("call_config0_1mb")
    fx = parity.load_golden("call_config0_1mb")
    _md_bams(monkeypatch)
    rows, log = tg._run_call_device(c, tmp_path, monkeypatch)
    gold = parity.golden_rows(fx)
    assert parity.rows_equal(rows, gold), parity.first_diff(rows, gold)
    assert log == fx["expected"]["log"]


def test_normcounts_worker_device_decode_md_config0(tmp_path, monkeypatch):
    """the drop-in get_callable_tricounts on the MD BAM of BASELINE configs[0] fills what it fills on the cs BAM"""
    c = cases.build_case("norm_config0_1mb")
    want = ts._run_norm(c, tmp_path, monkeypatch, "device")
    _md_bams(monkeypatch, "md_eqx")
    assert ts._run_norm(c, tmp_path, monkeypatch, "device") == want
    e = parity.load_golden("norm_config0_1mb")["expected"]
    ccs, rt, log, ties = want
    if not ties:
        assert all(ccs[t] == e["ccs_tri2count"].get(t, 0) for t in normcounts.TRI_LST) and log == e["log"]


@pytest.mark.parametrize("name", ["plain", "bq0_counts_deletions"])
def test_phase_edges_device_decode_md(tmp_path, monkeypatch, name):
    batch, hetsnp_lst, h2i, n, min_bq, min_mapq = te.mk.inputs(name)
    path = str(tmp_path / "e.bam")
    bamdec.write_batch_bam(path, "chr1", n, batch, tags="md")
    real = phaselib.edge_table
    monkeypatch.setattr(phaselib, "edge_table", lambda *a, **k: real(*a, **dict(k, decode="device")))
    edge_lst, e2c = phaselib.get_edges("chr1", path, min_bq, min_mapq, [h[0] for h in hetsnp_lst], hetsnp_lst, h2i)
    got = [[int(i), int(j)] + [int(v) for v in e2c[(i, j)]] for (i, j) in edge_lst]
    assert got == json.load(open(os.path.join(cases.GOLDEN_DIR, "edges.json")))["expected"][name]


def test_one_16mb_group_md_equals_cs(tmp_path):
    """one full decode group (worker.GROUP_SPAN) of a 30x contig: call, normcounts and the phase edges decoded on the
    device from the MD BAM give what they give from the cs BAM (each on a fresh context: nothing carried over)"""
    n = worker.GROUP_SPAN
    d = synth.generate(n, seed=5, copy=False)
    ref = bytes(d.ref)
    paths = {}
    for tags in ("cs", "md"):
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
                    res.append(caller.call_region(ctx, path, "chr1", loci, None, None, decode="device"))
                elif run == "norm":
                    res.append(normcounts.normcounts_region(ctx, path, "chr1", ref, loci, None, decode="device"))
                else:
                    res.append(phaselib.edge_table(ctx, path, "chr1", hpos, href, 10, 20, decode="device"))
        out[tags] = res
    _deep_equal(out["cs"], out["md"])


def _rows(rec):
    """site records as a sorted multiset: call_region returns them in the order the device wrote them, which is not
    fixed from one run to the next (the drop-in worker natsorts its rows)"""
    packed = rfn.repack_fields(rec[[n for n in rec.dtype.names if n != "pad0"]])
    return sorted(bytes(x) for x in packed.view(np.dtype((np.void, packed.dtype.itemsize))))


def _deep_equal(a, b):
    if isinstance(a, np.ndarray) and a.dtype.names:
        assert isinstance(b, np.ndarray) and a.dtype == b.dtype and _rows(a) == _rows(b)
    elif isinstance(a, np.ndarray):
        assert isinstance(b, np.ndarray) and a.shape == b.shape and np.array_equal(a, b)
    elif isinstance(a, (list, tuple)):
        assert type(a) is type(b) and len(a) == len(b)
        for x, y in zip(a, b):
            _deep_equal(x, y)
    elif isinstance(a, dict):
        assert a.keys() == b.keys()
        for k in a:
            _deep_equal(a[k], b[k])
    else:
        assert a == b
