"""Native BAM decoder (csrc/bamdec.c, include/himut_io.h) against the Python specification
(bamio.py + pack.py): same packed batch byte for byte, same fetch rule, same rejections."""
import ctypes as C
import os

import numpy as np
import pytest

import cases
from himut_b200 import bamdec, bamio, pack, synth


def _same(a, b):
    for name, _ in a._FIELDS:
        x, y = getattr(a, name), getattr(b, name)
        assert x.shape == y.shape and np.array_equal(x, y), name


def test_io_library_exports_every_declared_symbol():
    lib = C.CDLL(bamdec.lib_path())
    hdr = open(os.path.join(os.path.dirname(cases.GOLDEN_DIR), "..", "include", "himut_io.h")).read()
    import re
    declared = set(re.findall(r"\b(hm_(?:bam|bq)_\w+)\s*\(", hdr))
    assert declared == set(bamdec.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name


@pytest.mark.parametrize("threads", [1, 4])
def test_native_batch_equals_python_batch(tmp_path, threads):
    d = synth.generate(300_000, seed=11)
    path = str(tmp_path / "t.bam")
    bamio.write_batch_bam(path, "chr1", 300_000, d.batch)
    nb = bamdec.NativeBam(path, threads=threads)
    rd = bamio.BamReader(path)
    assert nb.references == rd.references and nb.lengths == rd.lengths and nb.header_text == rd.header_text
    qnames = {}  # the handle interns query names across windows; give the Python builder the same table
    for s, e in [(0, 300_000), (1, 200_000), (200_000, 299_998), (123_456, 123_457), (299_990, 300_000), (0, 1)]:
        bb = pack.BatchBuilder()
        bb.qnames = qnames
        _same(nb.read_batch("chr1", s, e), bamio.read_batch(rd, "chr1", s, e, builder=bb))
    whole = nb.read_batch("chr1", 0, 300_000)
    assert cases.batch_digest(whole) == cases.batch_digest(d.batch)
    assert nb.n_qnames() == len(set(d.batch.qname_id.tolist()))
    assert nb.qname(int(whole.qname_id[5])) == "read5"
    nb.close(); rd.close()


def test_qname_ids_are_stable_across_windows(tmp_path):
    d = synth.generate(200_000, seed=12)
    path = str(tmp_path / "t.bam")
    bamio.write_batch_bam(path, "chr1", 200_000, d.batch)
    nb = bamdec.NativeBam(path, threads=2)
    a = nb.read_batch("chr1", 0, 120_000)
    b = nb.read_batch("chr1", 100_000, 200_000)
    names_a = {nb.qname(int(i)) for i in a.qname_id}
    names_b = {nb.qname(int(i)) for i in b.qname_id}
    both = names_a & names_b
    assert both  # reads spanning the seam appear in both windows under the same id
    ids_a = {nb.qname(int(i)): int(i) for i in a.qname_id}
    ids_b = {nb.qname(int(i)): int(i) for i in b.qname_id}
    assert all(ids_a[n] == ids_b[n] for n in both)


def _write(path, records, reflen=1000):
    w = bamio.BamWriter(path, [("chr1", reflen), ("chr2", reflen)])
    for r in records:
        w.add(**r)
    w.close()


def _rec(pos=10, cigar=((0, 8),), seq="ACGTACGT", cs=":8", flag=0, qual=None, ref_id=0, qname="q", extra=()):
    tags = [("tp", "A", "P")] + ([("cs", "Z", cs)] if cs is not None else []) + list(extra)
    return dict(ref_id=ref_id, pos=pos, qname=qname, flag=flag, mapq=60, cigar=list(cigar), seq=seq,
                qual=bytes([40] * len(seq)) if qual is None else qual, tags=tags)


def test_soft_clips_secondary_supplementary_and_contigs(tmp_path):
    path = str(tmp_path / "m.bam")
    _write(path, [
        _rec(pos=10, cigar=((4, 2), (0, 6), (4, 1)), seq="NNACGTACN", cs=":6", qname="clip"),
        _rec(pos=12, flag=0x100, qname="secondary", cs=None),           # dropped before the cs lookup
        _rec(pos=14, flag=0x800, qname="supp", cs=":3*ag:2+tt-ca:0", cigar=((0, 6), (1, 2), (2, 2)), seq="ACGGACTT"),
        _rec(pos=20, cs="=ACGT*ct=CGT", seq="ACGTTCGT", qname="longform"),
        _rec(pos=5, ref_id=1, qname="other"),
    ])
    nb = bamdec.NativeBam(path, threads=1)
    rd = bamio.BamReader(path)
    qnames = {}
    for chrom in ("chr1", "chr2"):
        for s, e in [(0, 1000), (15, 16), (0, 11), (27, 40)]:
            bb = pack.BatchBuilder()
            bb.qnames = qnames
            _same(nb.read_batch(chrom, s, e), bamio.read_batch(rd, chrom, s, e, builder=bb))
    b = nb.read_batch("chr1", 0, 1000)
    assert [nb.qname(int(i)) for i in b.qname_id] == ["clip", "supp", "longform"]
    assert b.qstart.tolist() == [2, 0, 0] and b.qlen.tolist() == [9, 8, 8]


@pytest.mark.parametrize("bad", [
    dict(cs=None),                                      # KeyError in BAM.__init__
    dict(seq="ACNTACGT"),                               # N under a match
    dict(cs=":2*an:5"),                                 # substitution to N
    dict(cs=":9"),                                      # cs longer than the read
    dict(cs=":7"),                                      # cs / CIGAR span mismatch
    dict(cs=":4~gt12ag:4"),                             # intron token
    dict(qual=b"\xff" * 8),                             # missing qualities
])
def test_rejections_match_the_python_specification(tmp_path, bad):
    path = str(tmp_path / "b.bam")
    _write(path, [_rec(**bad)])
    nb = bamdec.NativeBam(path, threads=1)
    with pytest.raises(pack.BatchFormatError):
        nb.read_batch("chr1", 0, 1000)
    with pytest.raises(pack.BatchFormatError):
        bamio.read_batch(bamio.BamReader(path), "chr1", 0, 1000)


def test_without_index_and_empty_contig(tmp_path):
    d = synth.generate(60_000, seed=13)
    path = str(tmp_path / "t.bam")
    bamio.write_batch_bam(path, "chr1", 60_000, d.batch)
    os.remove(path + ".bai")
    nb = bamdec.NativeBam(path, threads=2)
    _same(nb.read_batch("chr1", 20_000, 30_000), bamio.read_batch(bamio.BamReader(path), "chr1", 20_000, 30_000))
    path2 = str(tmp_path / "e.bam")
    _write(path2, [_rec(ref_id=1)])
    nb2 = bamdec.NativeBam(path2)
    b = nb2.read_batch("chr1", 0, 1000)
    assert b.n_reads == 0 and b.seq.size == 16 and b.bq.size == 16


def test_native_writer_equals_python_writer(tmp_path):
    d = synth.generate(150_000, seed=14)
    p_py, p_c = str(tmp_path / "py.bam"), str(tmp_path / "c.bam")
    bamio.write_batch_bam(p_py, "chr1", 150_000, d.batch)
    bamdec.write_batch_bam(p_c, "chr1", 150_000, d.batch, threads=3)
    a, b = bamio.BamReader(p_py), bamio.BamReader(p_c)
    assert a.header_text == b.header_text and a.references == b.references and a.lengths == b.lengths
    key = lambda r: (r.query_name, r.reference_start, r.reference_end, r.flag, r.mapping_quality, r.tags.get("cs"), r.tags.get("tp"),
                     bytes(r.qual), bytes(r.seq_nibbles), r.query_alignment_start, r.query_alignment_end)
    for s, e in [(0, 150_000), (70_000, 70_001), (149_000, 150_000)]:
        assert [key(r) for r in a.fetch("chr1", s, e)] == [key(r) for r in b.fetch("chr1", s, e)]
    nb = bamdec.NativeBam(p_c, threads=2)
    assert cases.batch_digest(nb.read_batch("chr1", 0, 150_000)) == cases.batch_digest(d.batch)


def test_batch_without_base_stream(tmp_path):
    """HM_BAM_OPT_NO_SEQ: everything but seq / seq_off is what the full decode gives, the base checks stay"""
    d = synth.generate(200_000, seed=15, softclip_frac=0.2)
    path = str(tmp_path / "t.bam")
    bamio.write_batch_bam(path, "chr1", 200_000, d.batch)
    nb = bamdec.NativeBam(path, threads=2)
    full = nb.read_batch("chr1", 0, 200_000)
    bare = nb.read_batch("chr1", 0, 200_000, seq=False)
    assert bare.seq.size == 0 and bare.seq_off.size == 0
    s = bare.as_struct()
    assert s.seq is None and s.seq_off is None and s.seq_bytes == 0
    for name, _ in full._FIELDS:
        if name not in ("seq", "seq_off"):
            assert np.array_equal(getattr(full, name), getattr(bare, name)), name
    assert np.array_equal(nb.read_batch("chr1", 0, 200_000).seq, full.seq)  # and back
    # a base outside A/C/G/T under a cs match is still refused
    bad = str(tmp_path / "bad.bam")
    _write(bad, [_rec(pos=10, cigar=((0, 6),), seq="ACNTAC", cs=":6", qname="n_under_match")])
    nb2 = bamdec.NativeBam(bad, threads=1)
    with pytest.raises(pack.BatchFormatError):
        nb2.read_batch("chr1", 0, 1000, seq=False)


def test_base_conversion_at_every_length(tmp_path):
    """the decoder converts 4-bit bases 32 at a time and packs 2-bit codes 16 at a time with a scalar tail: records of
    every length from 1 to 150 with N / IUPAC letters in their soft clips must pack like the Python packer"""
    import random
    rnd = random.Random(9)
    recs = []
    for n in range(1, 151):
        lead, trail = rnd.randrange(0, 4), rnd.randrange(0, 4)
        m = max(1, n - lead - trail)
        clip = lambda k: "".join(rnd.choice("ACGTNRY") for _ in range(k))
        body = "".join(rnd.choice("ACGT") for _ in range(m))
        cigar = ([(4, lead)] if lead else []) + [(0, m)] + ([(4, trail)] if trail else [])
        recs.append(_rec(pos=10 + n, cigar=cigar, seq=clip(lead) + body + clip(trail), cs=":%d" % m, qname="r%d" % n))
    path = str(tmp_path / "len.bam")
    _write(path, recs)
    nb = bamdec.NativeBam(path, threads=2)
    bb = pack.BatchBuilder()
    got = nb.read_batch("chr1", 0, 1000)
    _same(got, bamio.read_batch(bamio.BamReader(path), "chr1", 0, 1000, builder=bb))
    assert got.n_reads == 150


@pytest.mark.parametrize("threads", [1, 3])
def test_compact_quality_stream_is_lossless_on_the_cpu(threads):
    """hm_bq_compact_build (host) against the format include/himut_b200.h specifies, expanded here with numpy the way
    k_bq_expand does on the device: bit set = modal value, clear bits take the exceptions read by read in base order"""
    from himut_b200 import synth
    import cases
    for batch in (synth.generate(300_000, seed=61).batch, cases.adversarial_batch(5, contig_len=6000, n_reads=300, max_len=2000)[0]):
        cq = bamdec.compact_bq(batch, threads=threads)
        assert cq.mask.size * 8 == batch.bq.size and cq.exc_off.size == batch.n_reads + 1
        bits = np.unpackbits(cq.mask, bitorder="little").astype(bool)
        vals, counts = np.unique(batch.bq[np.concatenate([np.arange(int(o), int(o) + int(l)) for o, l in zip(batch.bq_off, batch.qlen)])],
                                 return_counts=True)
        assert cq.modal == int(vals[np.argmax(counts)])
        out = np.zeros(batch.bq.size, np.uint8)
        for r in range(batch.n_reads):
            o, l = int(batch.bq_off[r]), int(batch.qlen[r])
            m = bits[o:o + l]
            seg = np.full(l, cq.modal, np.uint8)
            e0, e1 = int(cq.exc_off[r]), int(cq.exc_off[r + 1])
            assert e1 - e0 == int((~m).sum())
            seg[~m] = cq.exc[e0:e1]
            out[o:o + l] = seg
            pad_end = int(batch.bq_off[r + 1]) if r + 1 < batch.n_reads else batch.bq.size
            assert not bits[o + l:pad_end].any()      # padding bits are clear
            assert np.array_equal(seg, batch.bq[o:o + l])
        assert int(cq.exc_off[-1]) == cq.n_exc


def test_hard_clipped_records_are_decoded_as_pysam_presents_them(tmp_path):
    """SEQ holds no hard-clipped base; query_alignment_start counts soft clips only: the reference processes such
    records (minimap2 writes them for supplementary alignments), native decoder and specification agree"""
    path = str(tmp_path / "h.bam")
    _write(path, [
        _rec(pos=10, cigar=((5, 3), (0, 8)), qname="hard5"),
        _rec(pos=12, cigar=((5, 4), (4, 2), (0, 5), (4, 1), (5, 7)), seq="NNACGTAN", cs=":5", qname="hard_soft"),
    ])
    nb = bamdec.NativeBam(path, threads=1)
    rd = bamio.BamReader(path)
    bb = pack.BatchBuilder()
    got = nb.read_batch("chr1", 0, 1000)
    _same(got, bamio.read_batch(rd, "chr1", 0, 1000, builder=bb))
    assert got.qstart.tolist() == [0, 2] and got.qlen.tolist() == [8, 8] and got.tend.tolist() == [18, 17]


def _expand(batch, cq):
    """hm_bq_compact -> the one-byte-per-base stream (what k_bq_expand does on the device)"""
    out = np.zeros(batch.bq_bytes_expanded, np.uint8)
    bits = np.unpackbits(cq.mask, bitorder="little")
    for r in range(batch.n_reads):
        o, n = int(batch.bq_off[r]), int(batch.qlen[r])
        m = bits[o:o + n].astype(bool)
        q = np.full(n, cq.modal, np.uint8)
        e0, e1 = int(cq.exc_off[r]), int(cq.exc_off[r + 1])
        assert e1 - e0 == int((~m).sum())
        q[~m] = cq.exc[e0:e1]
        out[o:o + n] = q
        assert not bits[o + n:o + ((n + 15) & ~15)].any()  # padding bits are clear
    return out


@pytest.mark.parametrize("threads", [1, 4])
def test_compact_qualities_from_the_parse_pass(tmp_path, threads):
    """HM_BAM_OPT_COMPACT_BQ: the decoder writes bitmap + exceptions while it parses the records; expanded, they are
    the plain stream byte for byte; everything else in the batch is unchanged"""
    d = synth.generate(300_000, seed=21)
    path = str(tmp_path / "c.bam")
    bamio.write_batch_bam(path, "chr1", 300_000, d.batch)
    nb = bamdec.NativeBam(path, threads=threads)
    for s, e in [(0, 300_000), (120_000, 180_000), (299_990, 300_000)]:
        plain = nb.read_batch("chr1", s, e, seq=False)
        batch, cq = nb.read_batch("chr1", s, e, seq=False, compact=True)
        assert batch.bq.size == 0 and batch.bq_bytes_expanded == plain.bq.size
        assert np.array_equal(_expand(batch, cq), plain.bq)
        for name in ("tstart", "tend", "qstart", "qlen", "mapq", "flags", "qname_id", "bq_off", "op_off", "n_ops", "ops"):
            assert np.array_equal(getattr(batch, name), getattr(plain, name)), name
        assert cq.n_exc == int(cq.exc_off[-1]) and cq.mask.size * 8 == plain.bq.size
    nb.close()


def test_two_buffer_sets(tmp_path):
    """a batch decoded into one buffer set stays valid while the next is decoded into the other"""
    d = synth.generate(200_000, seed=22)
    path = str(tmp_path / "s.bam")
    bamio.write_batch_bam(path, "chr1", 200_000, d.batch)
    nb = bamdec.NativeBam(path, threads=2)
    want_a = nb.read_batch("chr1", 0, 100_000)
    want_b = nb.read_batch("chr1", 100_000, 200_000)
    a = nb.read_batch("chr1", 0, 100_000, copy=False, buffer_set=0)
    b = nb.read_batch("chr1", 100_000, 200_000, copy=False, buffer_set=1)
    assert cases.batch_digest(a) == cases.batch_digest(want_a)  # not overwritten by the second decode
    assert cases.batch_digest(b) == cases.batch_digest(want_b)
    a2, cq = nb.read_batch("chr1", 0, 100_000, copy=False, seq=False, compact=True, buffer_set=0)
    assert cases.batch_digest(b) == cases.batch_digest(want_b)
    assert np.array_equal(_expand(a2, cq), want_a.bq)
    nb.close()


def test_malformed_records_are_rejected_not_read_past(tmp_path):
    """fields taken from the file are checked against block_size before they are used: a corrupt record gives a
    BatchFormatError, never an out-of-bounds read (run under ASan by tools/sanitize_host.sh)"""
    import gzip
    import struct
    import zlib
    path = str(tmp_path / "ok.bam")
    _write(path, [_rec(pos=10, qname="first"), _rec(pos=20, qname="second", extra=[("xb", "B", ("c", [1, 2, 3]))])])
    raw = bytearray(gzip.open(path, "rb").read())  # BGZF members are gzip members
    first = raw.find(b"first\x00") - 36  # block_size field of the first record
    assert first > 0
    bs = struct.unpack_from("<I", raw, first)[0]
    rng = np.random.default_rng(5)

    def rewrite(mut, name):
        return _rebgzf(mut, str(tmp_path / name))

    cases_ = []
    m = bytearray(raw); struct.pack_into("<i", m, first + 4 + 16, 1 << 20); cases_.append(m)       # l_seq far past the record
    m = bytearray(raw); m[first + 4 + 8] = 255; cases_.append(m)                                    # l_name past the record
    m = bytearray(raw); struct.pack_into("<H", m, first + 4 + 12, 60000); cases_.append(m)          # n_cigar_op past the record
    m = bytearray(raw); struct.pack_into("<I", m, first, 16); cases_.append(m)                      # block_size below the fixed part
    m = bytearray(raw); m[first + 4 + bs - 1] = 65; cases_.append(m)                                # last tag string unterminated
    for k in range(40):                                                                             # random byte damage inside the record
        m = bytearray(raw)
        for _ in range(3):
            m[first + 4 + int(rng.integers(0, bs))] = int(rng.integers(0, 256))
        cases_.append(m)
    n_bad = 0
    for i, m in enumerate(cases_):
        p = rewrite(m, "mut%d.bam" % i)
        try:
            nb = bamdec.NativeBam(p, threads=1)
        except IOError:
            n_bad += 1
            continue
        try:
            nb.read_batch("chr1", 0, 1000)
            nb.read_batch("chr1", 0, 1000, seq=False, compact=True)
            nb.window_qlens("chr1", 0, 1000)
        except pack.BatchFormatError:
            n_bad += 1
        nb.close()
    assert n_bad >= 5  # the five structural mutations at least


def _rebgzf(raw, out):
    """an inflated BAM stream -> BGZF blocks (zlib) at `out`, without a BAI"""
    import struct
    import zlib
    blocks = []
    for i in range(0, len(raw), 60000):
        piece = bytes(raw[i:i + 60000])
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        comp = c.compress(piece) + c.flush()
        blocks.append(b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(comp) + 25) + comp +
                      struct.pack("<II", zlib.crc32(piece) & 0xffffffff, len(piece)))
    blocks.append(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
    with open(out, "wb") as f:
        f.write(b"".join(blocks))
    return out


def bad_b_subtype(tmp_path):
    """a record with a B array tag of subtype 'x' between cs:Z and another tag: htslib rejects such a record as
    corrupted aux data; a walker that took 'x' for 4-byte elements would step into the next tag"""
    import gzip
    path = str(tmp_path / "sub.bam")
    _write(path, [_rec(pos=10, qname="badsub", extra=[("xb", "B", ("C", [7])), ("yz", "Z", "abcdefgh")])])
    raw = gzip.open(path, "rb").read()
    assert raw.count(b"xbBC\x01\x00\x00\x00") == 1
    return _rebgzf(raw.replace(b"xbBC\x01\x00\x00\x00", b"xbBx\x01\x00\x00\x00"), str(tmp_path / "badsub.bam"))


B_SUBTYPE_MSG = "malformed BAM record badsub: truncated B tag or unknown B subtype (120)"


def test_unknown_b_subtype_is_rejected_by_every_walker(tmp_path):
    path = bad_b_subtype(tmp_path)
    nb = bamdec.NativeBam(path, threads=1)
    for kw in (dict(), dict(seq=False, compact=True)):
        with pytest.raises(pack.BatchFormatError) as ex:
            nb.read_batch("chr1", 0, 1000, **kw)
        assert str(ex.value) == B_SUBTYPE_MSG
    with pytest.raises(pack.BatchFormatError) as ex:
        nb.window_qlens("chr1", 0, 1000)
    assert str(ex.value) == B_SUBTYPE_MSG
    nb.close()
    with pytest.raises(bamio.BamError, match="unknown B subtype 'x'"):
        bamio.read_batch(bamio.BamReader(path), "chr1", 0, 1000)
