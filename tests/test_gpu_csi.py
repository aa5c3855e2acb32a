"""The device decoder on BAMs indexed with a CSI, and coordinates between 2^29 and 2^31 - 1 (where only a CSI can index a
contig) through every device path: the device batch against the host batch, `call_region` with and without --phase
against the oracle and the host-decoder run, `normcounts_region` against the oracle, and the phase edges against the
host edge table.  GPU."""
import numpy as np
import pytest

import cases
import parity
import test_gpu_bamdecode as tg
import test_gpu_bamdecode_seq as ts
import test_gpu_md_ops as tmd
from himut_b200 import abi, bamdec, bamio, caller, gtmodel, normcounts, phaselib, synth, worker
from oracle import oracle

pytestmark = pytest.mark.gpu

PARAMS = [(14, 5), (12, 6), (16, 4)]
LONG = 2**31 - 1
WINDOWS = [(0, 300_000), (1, 200_000), (200_000, 299_998), (123_456, 123_457), (299_990, 300_000), (0, 1), (300_005, 300_050)]


@pytest.mark.parametrize("writer", ["python", "native"])
@pytest.mark.parametrize("ms,depth", PARAMS)
def test_device_batch_equals_host_batch_through_a_csi(ctx, tmp_path, writer, ms, depth):
    n = 300_000
    d = synth.generate(n, seed=11)
    path = str(tmp_path / "t.bam")
    (bamio.write_batch_bam if writer == "python" else bamdec.write_batch_bam)(path, "chr1", n, d.batch, index="csi", min_shift=ms, depth=depth)
    nb = bamdec.NativeBam(path, threads=4)
    assert nb.index_kind == "csi"
    for s, e in WINDOWS:
        tg._same_as_host(ctx, nb, "chr1", s, e)
        ts._same_as_host(ctx, nb, "chr1", s, e)
    nb.close()


# ---------------------------------------------------------------------------------------------------- a contig of 2^31 - 1
N = 300_000


def _moved(batch, off, qoff):
    kw = {name: getattr(batch, name) for name, _ in abi.ReadBatch._FIELDS}
    kw["tstart"] = (batch.tstart.astype(np.int64) + off).astype(np.int32)
    kw["tend"] = (batch.tend.astype(np.int64) + off).astype(np.int32)
    kw["qname_id"] = batch.qname_id + np.uint32(qoff)
    return abi.ReadBatch(**kw)


@pytest.fixture(scope="module")
def long_contig(tmp_path_factory):
    """a 100 kb contig, then chrL of LN 2^31 - 1 with one 300 kb 30x stretch across 2^29, one across 2^30 and one whose
    last read ends at the contig's last base; the reference is N outside the stretches -> (path, loci, ref, phase
    table, chunk sets, hetSNPs)"""
    d = synth.generate(N, seed=71)
    small = synth.generate(100_000, seed=72)
    offs = [2**29 - N // 2, 2**30 - N // 2, LONG - int(d.batch.tend.max())]
    path = str(tmp_path_factory.mktemp("long") / "long.bam")
    w = bamio.BamWriter(path, [("chrS", 100_000), ("chrL", LONG)], index="csi")
    bamio._add_batch(w, 0, small.batch)
    for k, off in enumerate(offs):
        bamio._add_batch(w, 1, _moved(d.batch, off, 1_000_000 * (k + 1)))
    w.close()
    ref = bytearray(b"N") * LONG
    loci, hpos, href, halt, hbit, set_off = [], [], [], [], [], [0]
    het = d.germ["gt"] < 2
    gpos = d.germ["pos"][het].astype(np.int64)
    for off in offs:
        ref[off:off + N] = bytes(d.ref)
        for s, e in cases.chunkloci(0, N):
            loci.append(("chrL", s + off, e + off))
            m = (gpos >= s) & (gpos < e)
            hpos += (gpos[m] + off).tolist()
            href += d.germ["ref"][het][m].tolist()
            halt += d.germ["alt"][het][m].tolist()
            hbit += (d.germ["gt"][het][m] == 0).astype(np.uint8).tolist()
            set_off.append(len(hpos))
    assert int(d.batch.tend.max()) + offs[2] == LONG
    phase = dict(hpos=np.array(hpos, np.int32), href=np.array(href, np.uint8), halt=np.array(halt, np.uint8),
                 hbit=np.array(hbit, np.uint8), set_off=np.array(set_off, np.uint64))
    return path, loci, bytes(ref), phase, list(range(len(loci))), offs


def test_long_contig_device_batch_equals_host_batch(ctx, long_contig):
    path, _loci, _ref, _phase, _sets, offs = long_contig
    nb = bamdec.NativeBam(path, threads=4)
    assert nb.index_kind == "csi" and nb.lengths == [100_000, LONG]
    for chrom, s, e in [("chrS", 0, 100_000), ("chrL", 0, LONG), ("chrL", 2**29 - 1, 2**29 + 1), ("chrL", 2**30, 2**30 + 1),
                        ("chrL", LONG - 1, LONG), ("chrL", offs[0], offs[0] + N), ("chrL", offs[1] - 5, offs[1] + N // 3),
                        ("chrL", offs[2], LONG), ("chrL", 2**29 + 2 * N, 2**30 - 2 * N)]:
        got = tg._same_as_host(ctx, nb, chrom, s, e)
        ts._same_as_host(ctx, nb, chrom, s, e)
        if (chrom, s, e) == ("chrL", LONG - 1, LONG):
            assert got.n_reads > 0 and int(got.tend.max()) == LONG
    whole = nb.read_batch("chrL", 0, LONG, seq=False)
    assert (whole.tstart < 2**29).any() and (whole.tend > 2**29).any() and ((whole.tstart < 2**30) & (whole.tend > 2**30)).any()
    nb.close()


def _params(phase):
    return gtmodel.make_params(**dict(gtmodel.DEFAULT_CALL_ARGS, phase=phase))


def _base(phase, long_contig):
    """the oracle on the unshifted contig (the stretches' reads at offset 0, their hetSNPs as the stretches' phase
    sets): each stretch of chrL must give exactly this, moved by its offset"""
    _path, loci, _ref, table, sets, offs = long_contig
    d = synth.generate(N, seed=71)
    k = len(loci) // len(offs)
    local = [(s - offs[0], e - offs[0]) for _c, s, e in loci[:k]]
    n_h = int(table["set_off"][k])
    ph = dict(table, hpos=table["hpos"][:n_h] - offs[0], set_off=table["set_off"][:k + 1]) if phase else None
    for key in ("href", "halt", "hbit"):
        if phase:
            ph[key] = table[key][:n_h]
    return d, local, ph, k


@pytest.mark.parametrize("phase", [False, True])
def test_long_contig_call_region(ctx, long_contig, phase):
    """call_region on the device decoder equals the host-decoder run, and each stretch equals the oracle's records of
    the unshifted reads moved by the stretch's offset"""
    path, loci, _ref, table, sets, offs = long_contig
    p = _params(phase)
    out = {}
    for decode in ("device", "host"):
        ctx.set_params(p)
        ctx.set_site_sets()
        if phase:
            ctx.set_phase_sets(table)
        out[decode] = caller.call_region(ctx, path, "chrL", loci, sets if phase else None, phase, decode=decode)
    tmd._deep_equal(out["device"], out["host"])
    rec = parity.sort_records(out["device"][0])
    d, local, ph, k = _base(phase, long_contig)
    base, _log = oracle.call_chunks(p, d.batch, d.batch.chunk_table(local, list(range(k)) if phase else None), phase=ph)
    base = parity.sort_records(base)
    assert base.size > 100
    for j, off in enumerate(offs):
        part = rec[(rec["tpos"] >= off) & (rec["tpos"] < off + N)].copy()
        moved = base.copy()
        moved["tpos"] += off
        for x in (part, moved):  # chunk and phase-set numbers count from the stretch's first chunk in `base`
            x["chunk"] = 0
            x["phase_set"] = x["phase_set"] >= 0
        ok, why = parity.records_equal(parity.sort_records(part), parity.sort_records(moved))
        assert ok, (off, why)
    assert rec.size == 3 * base.size


def test_long_contig_normcounts_region(ctx, long_contig):
    """normcounts_region on the device decoder equals the host-decoder run and three times the oracle's counts of the
    unshifted contig (the reference outside the stretches is N)"""
    path, loci, ref, _table, _sets, offs = long_contig
    p = _params(False)
    out = {}
    for decode in ("device", "host"):
        ctx.set_params(p)
        ctx.set_site_sets()
        out[decode] = normcounts.normcounts_region(ctx, path, "chrL", ref, loci, None, decode=decode)
    for x, y in zip(out["device"], out["host"]):
        assert np.array_equal(np.asarray(x), np.asarray(y))
    d, local, _ph, _k = _base(False, long_contig)
    o = oracle.normcounts_chunks(p, d.batch, bytes(d.ref), d.batch.chunk_table(local))
    g = out["device"]
    assert np.array_equal(g[0], 3 * o[0]) and np.array_equal(g[1], 3 * o[1]) and g[3] == 3 * o[3]
    assert int(np.asarray(g[0]).sum()) > 0


def test_long_contig_phase_edges(ctx, long_contig):
    path, _loci, _ref, table, _sets, _offs = long_contig
    hpos, href = table["hpos"], table["href"]
    assert int(hpos.max()) > 2**30
    dev = phaselib.edge_table(ctx, path, "chrL", hpos, href, 10, 20, decode="device")
    host = phaselib.edge_table(ctx, path, "chrL", hpos, href, 10, 20, decode="host")
    assert np.array_equal(dev, host) and int(dev.sum()) > 0


def test_64mb_contig_csi_only_auto_takes_the_device(ctx, tmp_path, monkeypatch):
    """the 64 Mb contig written with a CSI only: call_region(decode="auto") decodes on the device and its records equal
    the same run on the BAI copy"""
    n = 64_000_000
    d = synth.generate(n, seed=5, copy=False)
    bai, csi = str(tmp_path / "b.bam"), str(tmp_path / "c.bam")
    bamdec.write_batch_bam(bai, "chr1", n, d.batch)
    bamdec.write_batch_bam(csi, "chr1", n, d.batch, index="csi")
    del d
    loci = [("chr1", s, e) for s, e in cases.chunkloci(0, n)]
    seen = ts._spy_decodes(monkeypatch)
    out = {}
    for path in (bai, csi):
        ctx.set_params(_params(False))
        ctx.set_site_sets()
        before = len(seen)
        out[path] = caller.call_region(ctx, path, "chr1", loci, None, False, decode="auto")
        assert len(seen) - before == len(worker.group_chunks(loci)) and all(tg.DECODE_KERNELS <= k for k, _ in seen[before:])
    assert bamdec.NativeBam(csi).index_kind == "csi"
    tmd._deep_equal(out[csi], out[bai])
