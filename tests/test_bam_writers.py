"""BAMs as other writers leave them, through every decoder of the package.

RecodedWriter compresses each BGZF block with deflate_enc.py instead of zlib, a different construct mix per block
(dynamic blocks whose code-length runs cross the literal / distance boundary, long codes, fixed blocks, empty stored
blocks, padding bits set), can put another gzip extra subfield before BC, leaves empty BGZF blocks between data
blocks (as concatenated BAMs have them) and cuts blocks inside records: inside block_size and inside the fixed 32
bytes.  hifi_tags gives each record the aux tags pbmm2 / minimap2 HiFi records carry, in every integer width, f, H, and
B arrays of every subtype (empty ones too; kinetics as long as the read, so records pass 64 KB and span blocks).

The same reads written plainly (zlib, cs / MD and tp only) and recoded with those tags must give the same batch from
the host decoder (plain and compact), the pure-Python reader, the device decoder (with and without bases), the same
window_qlens, and the same worker outputs on the GPU."""
import gzip
import random
import struct
import zlib

import numpy as np
import pytest

import cases
import deflate_enc as de
import parity
from himut_b200 import bamdec, bamio, synth

CHROM, N = "chr1", 120_000
REGIONS = [(0, N), (1, N // 3), (N // 3, N // 2), (N // 2, N // 2 + 1), (N - 2000, N), (40_000, 41_000)]
STRADDLE = (None, 1, 3, 4, 5, 20, 35, 36, 37, None, 2000)  # block ends this far into the next record (4 + 32: the fixed part)


def hifi_tags(rnd, l_seq, kinetics):
    """(tags before cs / MD, tags after it)"""
    before = [("NM", "C", rnd.randrange(256)), ("AS", "S", rnd.randrange(65536)), ("nn", "c", rnd.randrange(-128, 128)),
              ("de", "f", rnd.random() / 50), ("zm", "I", rnd.randrange(1 << 32)), ("sn", "B", ("f", [rnd.random() * 20 for _ in range(4)])),
              ("MM", "Z", "C+m?,%d;" % rnd.randrange(9)), ("ML", "B", ("C", [rnd.randrange(256) for _ in range(rnd.randrange(0, 3))])),
              ("xh", "H", "1AE3%02X" % rnd.randrange(256)), ("xe", "B", ("I", []))]
    after = [("rq", "f", 0.999), ("ys", "s", -rnd.randrange(1, 30000)), ("yi", "i", -rnd.randrange(1 << 31)),
             ("yc", "B", ("c", [-1, 2, -128])), ("yS", "B", ("s", [])), ("yI", "B", ("i", [-3, 1 << 30])), ("yF", "B", ("f", []))]
    if kinetics:
        g = np.random.default_rng(rnd.randrange(1 << 30))
        kin = lambda hi: np.minimum(g.exponential(12, l_seq), hi).astype(int).tolist()
        after = [("fi", "B", ("C", kin(255))), ("fp", "B", ("S", kin(65535))), ("ri", "B", ("C", kin(255))),
                 ("rp", "B", ("S", kin(65535)))] + after
    return before, after


def _recipe(k, chunk):
    """the blocks of BGZF block k's DEFLATE stream"""
    if not chunk:
        return [{"type": "stored", "data": b"", "pad": 0x7f}]
    a, b = len(chunk) // 3, 2 * len(chunk) // 3
    kind = k % 5
    if kind == 0:  # every symbol has a code; the 9-bit lengths run on from the last literal/length into the distances
        return [{"type": "dynamic", "tokens": de.tokenize(chunk), "combined": True, "lit_lens": [8] * 226 + [9] * 60,
                 "dist_lens": [9] * 8 + [6] * 5 + [5] * 13 + [3] * 4}]
    if kind == 1:
        return [{"type": "fixed", "tokens": de.tokenize(chunk)}]
    if kind == 2:
        return [{"type": "dynamic", "tokens": de.tokenize(chunk[:a]), "combined": True}, {"type": "stored", "data": b"", "pad": 0x55},
                {"type": "fixed", "tokens": de.tokenize(chunk[:b], a)}, {"type": "dynamic", "tokens": de.tokenize(chunk, b), "skew": True}]
    if kind == 3:
        return [{"type": "dynamic", "tokens": de.tokenize(chunk), "skew": True, "hclen": 19}]
    return [{"type": "stored", "data": chunk[:a], "pad": 0x7f}, {"type": "fixed", "tokens": de.tokenize(chunk, a)}]


class RecodedWriter(bamio.BamWriter):
    """bamio.BamWriter with deflate_enc blocks, chosen block ends, empty blocks and extra tags (see the module text);
    its BAI stays exact: the pending bytes always start the next block and are fewer than that block will hold"""

    def __init__(self, path, references, tags=True, extra_subfield=True, empty_every=7, straddle=STRADDLE, **kw):
        self.tags, self.extra_subfield, self.empty_every, self.straddle = tags, extra_subfield, empty_every, straddle
        self.cut, self.n_blocks, self.n_rec, self.census = 0xFF00, 0, 0, {}
        self.rnd = random.Random(17)
        super().__init__(path, references, **kw)

    def _emit_block(self, chunk):
        comp, data, census = de.encode(_recipe(self.n_blocks, chunk))
        xtra = b"XY\x03\x00abc" if self.extra_subfield else b""
        if 12 + 6 + len(xtra) + len(comp) + 8 > 65536:  # does not shrink: stored, as encoders do
            comp, data, census = de.encode([{"type": "stored", "data": chunk}])
        assert data == chunk and zlib.decompress(comp, -15) == chunk
        for key, v in census.items():
            self.census[key] = self.census.get(key, 0) + v
        xlen = len(xtra) + 6
        block = (b"\x1f\x8b\x08\x04\0\0\0\0\0\xff" + struct.pack("<H", xlen) + xtra + b"BC\x02\x00"
                 + struct.pack("<H", 12 + xlen + len(comp) + 8 - 1) + comp + struct.pack("<II", zlib.crc32(chunk), len(chunk)))
        self.f.write(block)
        self.coff += len(block)
        self.n_blocks += 1

    def _flush(self, everything=True):
        while len(self.buf) >= self.cut or (everything and self.buf):
            chunk = bytes(self.buf[:self.cut])
            del self.buf[:self.cut]
            self.cut = 0xFF00
            self._emit_block(chunk)
            if self.empty_every and self.n_blocks % self.empty_every == 0:
                self._emit_block(b"")

    def add(self, ref_id, pos, qname, flag, mapq, cigar, seq, qual, tags):
        off = self.straddle[self.n_rec % len(self.straddle)]
        if off is not None and len(self.buf) + off <= 0xFF00:
            self.cut = len(self.buf) + off
        self.n_rec += 1
        if self.tags:
            before, after = hifi_tags(self.rnd, len(seq), kinetics=self.n_rec % 3 != 1)
            tags = before + tags + after
        super().add(ref_id, pos, qname, flag, mapq, cigar, seq, qual, tags)


def write_recoded(path, chrom, contig_len, batch, tags="cs", **kw):
    """write_batch_bam's records through RecodedWriter -> the writer"""
    w = RecodedWriter(path, [(chrom, contig_len)], **kw)
    bamio._add_batch(w, 0, batch, tags)
    w.close()
    return w


@pytest.fixture(scope="module")
def bams(tmp_path_factory):
    """per tag form: the plain zlib BAM and the recoded one with the HiFi tags, of the same reads (10-60 kb)"""
    d = synth.generate(N, seed=41, read_len_min=10_000, read_len_max=60_000, read_len_mean=25_000, read_len_sd=12_000, depth=4.0)
    out = {}
    for form in ("cs", "md"):
        p = str(tmp_path_factory.mktemp(form))
        plain, rec = p + "/plain.bam", p + "/recoded.bam"
        bamio.write_batch_bam(plain, CHROM, N, d.batch, tags=form)
        w = write_recoded(rec, CHROM, N, d.batch, tags=form)
        out[form] = (plain, rec, w)
    return d, out


def test_the_recoded_file_has_what_it_should(bams):
    """the constructs, the record sizes, the empty blocks, the extra subfield and the straddles are really there"""
    d, out = bams
    _plain, rec, w = out["cs"]
    for key in ("rle16_cross", "stored_empty_middle", "stored_pad_nonzero", "fixed", "hclen_19", "hlit_286"):
        assert w.census.get(key), key
    assert max(k for k in range(16) if w.census.get("dynamic.ll_len_%d" % k)) >= 13
    assert int(d.batch.qlen.min()) > 9_000 and int(d.batch.qlen.max()) > 40_000
    raw = open(rec, "rb").read()
    sizes, p, n_empty = [], 0, 0
    assert raw.endswith(bamio._BGZF_EOF)
    while p < len(raw) - len(bamio._BGZF_EOF):
        xlen = struct.unpack_from("<H", raw, p + 10)[0]
        assert xlen == 13 and raw[p + 12:p + 14] == b"XY"
        bsize = struct.unpack_from("<H", raw, p + 12 + xlen - 2)[0] + 1
        isize = struct.unpack_from("<I", raw, p + bsize - 4)[0]
        n_empty += isize == 0
        sizes.append(isize)
        p += bsize
    assert n_empty >= 3
    data = gzip.decompress(raw)  # BGZF blocks are gzip members
    q = 12 + struct.unpack_from("<i", data, 4)[0]
    for _ in range(struct.unpack_from("<i", data, q - 4)[0]):
        q += 8 + struct.unpack_from("<i", data, q)[0]
    starts = []
    while q < len(data):
        starts.append(q)
        q += 4 + struct.unpack_from("<i", data, q)[0]
    ends = set(np.cumsum(sizes).tolist())
    into = {o for st in starts for o in range(1, 37) if st + o in ends}
    assert into & {1, 2, 3} and into & set(range(4, 36))  # inside block_size, inside the fixed 32 bytes
    rd = bamio.BamReader(rec)
    big = [r for r in rd.fetch(CHROM) if len(r.qual) * 7 > 65280]
    assert big and len(sizes) > 3 * len(big)
    rd.close()


def _host(path, s, e, **kw):
    nb = bamdec.NativeBam(path, threads=2)
    try:
        return nb.read_batch(CHROM, s, e, **kw)
    finally:
        nb.close()


@pytest.mark.parametrize("form", ["cs", "md"])
def test_host_and_python_batches_do_not_see_the_tags_or_the_encoding(bams, form):
    d, out = bams
    plain, rec, _w = out[form]
    nb_p, nb_r = bamdec.NativeBam(plain, threads=3), bamdec.NativeBam(rec, threads=3)
    rd_p, rd_r = bamio.BamReader(plain), bamio.BamReader(rec)
    for s, e in REGIONS:
        want = nb_p.read_batch(CHROM, s, e)
        assert cases.batch_digest(nb_r.read_batch(CHROM, s, e)) == cases.batch_digest(want), (s, e)
        a, ca = nb_p.read_batch(CHROM, s, e, seq=False, compact=True)
        b, cb = nb_r.read_batch(CHROM, s, e, seq=False, compact=True)
        assert cases.batch_digest(a) == cases.batch_digest(b)
        assert ca.modal == cb.modal and all(np.array_equal(getattr(ca, f), getattr(cb, f)) for f in ("mask", "exc", "exc_off"))
        py_p, py_r = bamio.read_batch(rd_p, CHROM, s, e), bamio.read_batch(rd_r, CHROM, s, e)
        assert cases.batch_digest(py_r) == cases.batch_digest(py_p), (s, e)
        assert nb_r.window_qlens(CHROM, s, e).tolist() == nb_p.window_qlens(CHROM, s, e).tolist()
    whole = nb_r.read_batch(CHROM, 0, N)
    assert whole.n_reads == d.batch.n_reads
    for h in (nb_p, nb_r, rd_p, rd_r):
        h.close()


def test_python_reader_sees_every_tag_type(tmp_path):
    """the values BamWriter.add packs come back from the record bytes as written"""
    path = str(tmp_path / "t.bam")
    rnd = random.Random(3)
    before, after = hifi_tags(rnd, 12, kinetics=True)
    w = bamio.BamWriter(path, [(CHROM, 1000)])
    w.add(0, 10, "q", 0, 60, [(0, 12)], "ACGTACGTACGT", bytes([30] * 12), before + [("cs", "Z", ":12"), ("tp", "A", "P")] + after)
    w.close()
    rd = bamio.BamReader(path)
    (r,) = list(rd.fetch(CHROM))
    assert r.tags == {"cs": ":12", "tp": "P"}
    raw = gzip.open(path, "rb").read()
    for tag, ty, val in before + after:
        k = raw.index(tag.encode() + ty.encode())
        if ty == "B":
            sub, vals = val
            assert raw[k + 3:k + 4] == sub.encode() and struct.unpack_from("<I", raw, k + 4)[0] == len(vals)
            got = struct.unpack_from("<%d%s" % (len(vals), bamio._TAG_FMT[sub]), raw, k + 8)
            assert np.allclose(got, vals, rtol=1e-6) if sub == "f" else list(got) == vals
        elif ty not in "ZHA":
            got = struct.unpack_from("<" + bamio._TAG_FMT[ty], raw, k + 3)[0]
            assert abs(got - val) < 1e-6 * max(1, abs(val)) if ty == "f" else got == val
    with pytest.raises(ValueError):
        bamio.BamWriter(str(tmp_path / "x.bam"), [(CHROM, 1000)]).add(0, 1, "q", 0, 60, [(0, 1)], "A", b"\x1e", [("xx", "q", 1)])


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["cs", "md"])
def test_device_batches_do_not_see_the_tags_or_the_encoding(ctx, bams, form):
    import test_gpu_bamdecode as tg
    import test_gpu_bamdecode_seq as tsq
    _d, out = bams
    plain, rec, _w = out[form]
    nb_p, nb_r = bamdec.NativeBam(plain, threads=2), bamdec.NativeBam(rec, threads=2)
    for s, e in REGIONS:
        got = tg._same_as_host(ctx, nb_r, CHROM, s, e)
        assert cases.batch_digest(got) == cases.batch_digest(tg._same_as_host(ctx, nb_p, CHROM, s, e))
        tsq._same_as_host(ctx, nb_r, CHROM, s, e)
    nb_p.close()
    nb_r.close()


def _recoded_inputs(monkeypatch):
    """the workers' test BAMs (test_gpu_worker._inputs) written by RecodedWriter with the HiFi tags"""
    monkeypatch.setattr(bamio, "write_batch_bam", lambda path, chrom, n, batch, **k: write_recoded(path, chrom, n, batch, **k))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["call_basic", "call_phase_indel", "call_adversarial_b"])
def test_call_worker_on_recoded_tagged_bams(name, tmp_path, monkeypatch):
    import test_gpu_bamdecode as tg
    _recoded_inputs(monkeypatch)
    c = cases.build_case(name)
    fx = parity.load_golden(name)
    rows, log = tg._run_call_device(c, tmp_path, monkeypatch)
    gold = parity.golden_rows(fx)
    assert parity.rows_equal(rows, gold), parity.first_diff(rows, gold)
    assert log == fx["expected"]["log"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["norm_basic", "norm_phase"])
def test_normcounts_worker_on_recoded_tagged_bams(name, tmp_path, monkeypatch):
    import test_gpu_bamdecode_seq as tsq
    c = cases.build_case(name)
    want = tsq._run_norm(c, tmp_path, monkeypatch, "device")
    _recoded_inputs(monkeypatch)
    seen = tsq._spy_decodes(monkeypatch)
    assert tsq._run_norm(c, tmp_path, monkeypatch, "device") == want
    assert seen


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["plain", "bq0_counts_deletions"])
def test_phase_edges_on_recoded_tagged_bams(tmp_path, monkeypatch, name):
    import json
    import os
    import test_edges as te
    from himut_b200 import phaselib, worker
    batch, hetsnp_lst, h2i, n, min_bq, min_mapq = te.mk.inputs(name)
    path = str(tmp_path / "e.bam")
    write_recoded(path, "chr1", n, batch)
    monkeypatch.setattr(worker, "GROUP_SPAN", 37_000)
    real = phaselib.edge_table
    monkeypatch.setattr(phaselib, "edge_table", lambda *a, **k: real(*a, **dict(k, decode="device")))
    edge_lst, e2c = phaselib.get_edges("chr1", path, min_bq, min_mapq, [h[0] for h in hetsnp_lst], hetsnp_lst, h2i)
    got = [[int(i), int(j)] + [int(v) for v in e2c[(i, j)]] for (i, j) in edge_lst]
    assert got == json.load(open(os.path.join(cases.GOLDEN_DIR, "edges.json")))["expected"][name]
