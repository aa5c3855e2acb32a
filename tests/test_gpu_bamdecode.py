"""Device BAM decoder (bamgpu.cuh, hm_decode_bam_*): k_bgzf_inflate against zlib, the resident batch against the host
decoder's no-seq batch byte for byte, the host decoder's rejections and messages, and the `call` worker on the device
path against the reference's outputs.  GPU."""
import gzip
import os
import struct
import zlib

import numpy as np
import pytest

import cases
import parity
import test_bam_plan as tp
import test_bamdec as tb
import test_gpu_worker as tw
import test_inflate as ti
from himut_b200 import bamdec, bamio, caller, lib, pack, synth, worker

pytestmark = pytest.mark.gpu

DECODE_KERNELS = {"k_bgzf_inflate", "k_bam_walk", "k_bam_select", "k_bam_parse"}


@pytest.mark.parametrize("level", [0, 1, 6, 9])
@pytest.mark.parametrize("strategy", [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE])
def test_device_inflate_matches_zlib(ctx, level, strategy):
    for data in ti._payloads():
        data = data[:65536]
        comp = ti._raw_deflate(data, level, strategy)
        rc, got = ctx.inflate_test(comp, len(data), zlib.crc32(data))
        assert rc == 0 and got == data, (level, strategy, len(data))


def test_device_inflate_rejects_truncated_and_flipped_streams(ctx):
    """200 single-bit flips and every truncation class: an error code, or (a flip in bits the stream ignores) the
    right bytes — never a wrong result"""
    rng = np.random.default_rng(3)
    data = b"".join(ti._payloads())[:60000]
    comp = ti._raw_deflate(data, 6)
    crc = zlib.crc32(data)
    for cut in (0, 1, 2, len(comp) // 3, len(comp) // 2, len(comp) - 1):
        rc, _ = ctx.inflate_test(comp[:cut], len(data), crc)
        assert rc != 0
    rc, _ = ctx.inflate_test(comp, len(data) - 1, crc)  # output that is not exactly ISIZE
    assert rc != 0
    rc, _ = ctx.inflate_test(comp, len(data) + 1, crc)
    assert rc != 0
    for _ in range(200):
        m = bytearray(comp)
        bit = int(rng.integers(0, 8 * len(m)))
        m[bit >> 3] ^= 1 << (bit & 7)
        rc, got = ctx.inflate_test(bytes(m), len(data), crc)
        assert rc != 0 or got == data
    far = b"\x01" + bytes([0x08, 0x00, 0xf7, 0xff]) + b"abcd"  # stored block whose LEN runs past the input
    assert ctx.inflate_test(far, 8, zlib.crc32(b"abcdabcd"))[0] != 0
    # fixed-code block: literal 'a', then length 3 at distance 2 (only one byte out so far), then end of block
    bits = "1" + "10"  # BFINAL, BTYPE = 01 (LSB first)
    bits += format(0x30 + ord("a"), "08b")  # literal 'a' (8-bit code, MSB first)
    bits += format(1, "07b")  # length code 257 (= 3)
    bits += format(1, "05b")  # distance code 1 (= 2)
    bits += format(0, "07b")  # end of block
    raw = bytearray((len(bits) + 7) // 8)
    for i, b in enumerate(bits):
        raw[i >> 3] |= int(b) << (i & 7)
    assert ctx.inflate_test(bytes(raw), 4, 0)[0] != 0


def _device_batch(ctx, nb, chrom, s, e):
    r = ctx.decode_region(nb, chrom, s, e)
    ran = {k for k, _ in ctx.last_decode_times}
    assert "k_bgzf_inflate" in ran and (r.n_reads == 0 or DECODE_KERNELS <= ran)
    b = ctx.read_back()
    assert b.n_reads == r.n_reads and np.array_equal(b.tstart, r.tstart) and np.array_equal(b.tend, r.tend)
    return b


def _same_as_host(ctx, nb, chrom, s, e):
    want = nb.read_batch(chrom, s, e, seq=False)
    got = _device_batch(ctx, nb, chrom, s, e)
    for name in ("tstart", "tend", "qstart", "qlen", "mapq", "qname_id", "bq_off", "op_off", "n_ops", "bq", "ops"):
        x, y = getattr(got, name), getattr(want, name)
        assert x.shape == y.shape and np.array_equal(x, y), (name, chrom, s, e)
    return got


def _write_level(path, parts, writer, level):
    if writer == "native":
        bamdec.write_batch_bam(path, parts[0][0], parts[0][1], parts[0][2], level=level)
    else:
        w = bamio.BamWriter(path, [(c, n) for c, n, _ in parts], level=level)
        for rid, (_c, _n, b) in enumerate(parts):
            bamio._add_batch(w, rid, b)
        w.close()


@pytest.mark.parametrize("writer", ["python", "native"])
@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_device_batch_equals_host_batch(ctx, tmp_path, writer, level):
    n = 300_000
    d = synth.generate(n, seed=11)
    path = str(tmp_path / "t.bam")
    _write_level(path, [("chr1", n, d.batch)], writer, level)
    nb = bamdec.NativeBam(path, threads=4)
    for s, e in [(0, n), (1, 200_000), (200_000, 299_998), (123_456, 123_457), (299_990, n), (0, 1), (n + 5, n + 50)]:
        _same_as_host(ctx, nb, "chr1", s, e)
    nb.close()


def test_device_batch_soft_clips_secondary_supplementary_contigs(ctx, tmp_path):
    path = str(tmp_path / "m.bam")
    tb._write(path, [
        tb._rec(pos=10, cigar=((4, 2), (0, 6), (4, 1)), seq="NNACGTACN", cs=":6", qname="clip"),
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
    nb.close()


def test_device_batch_multi_contig_and_without_index(ctx, tmp_path):
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


def test_device_batch_of_the_64mb_contig(ctx, tmp_path):
    """the contig of tools/worker_trace.py (64 Mb, 30x, seed 5): whole, and per 16 Mb group"""
    n = 64_000_000
    d = synth.generate(n, seed=5, copy=False)
    path = str(tmp_path / "c.bam")
    bamdec.write_batch_bam(path, "chr1", n, d.batch)
    del d
    nb = bamdec.NativeBam(path)
    for s, e in [(0, n)] + [(g, g + 16_000_000) for g in range(0, n, 16_000_000)]:
        _same_as_host(ctx, nb, "chr1", s, e)
    nb.close()


def _device_error(ctx, path, s=0, e=1000):
    nb = bamdec.NativeBam(path, threads=1)
    try:
        with pytest.raises(pack.BatchFormatError) as ex:
            ctx.decode_region(nb, "chr1", s, e)
        return str(ex.value)
    finally:
        nb.close()


def _host_error(path, s=0, e=1000):
    nb = bamdec.NativeBam(path, threads=1)
    try:
        with pytest.raises(pack.BatchFormatError) as ex:
            nb.read_batch("chr1", s, e, seq=False)
        return str(ex.value)
    finally:
        nb.close()


@pytest.mark.parametrize("bad", [
    dict(cs=None), dict(seq="ACNTACGT"), dict(cs=":2*an:5"), dict(cs=":9"), dict(cs=":7"), dict(cs=":4~gt12ag:4"),
    dict(qual=b"\xff" * 8),
])
def test_device_rejections_match_the_host(ctx, tmp_path, bad):
    path = str(tmp_path / "b.bam")
    tb._write(path, [tb._rec(**bad)])
    assert _device_error(ctx, path) == _host_error(path)


def test_device_rejects_an_unknown_b_subtype_as_the_host_does(ctx, tmp_path):
    path = tb.bad_b_subtype(tmp_path)
    assert _device_error(ctx, path) == _host_error(path) == tb.B_SUBTYPE_MSG


def test_device_reports_the_record_the_host_reports(ctx, tmp_path):
    """a bad cs string (found when records are decoded) before a record without cs (found when they are selected): the
    host decoder selects every record of its buffer before it decodes any, so it names the second record; so does the
    device decoder"""
    path = str(tmp_path / "two.bam")
    tb._write(path, [tb._rec(pos=10, cs=":7", qname="badcs"), tb._rec(pos=20, cs=None, qname="nocs")])
    msg = _host_error(path)
    assert msg.startswith("nocs has no cs:Z tag")
    assert _device_error(ctx, path) == msg


def test_device_ignores_a_corrupt_block_past_the_region(ctx, tmp_path):
    """the plan ends at the region's end: a damaged block far past it is never copied or inflated, as the host
    decoder never reads it"""
    n = 300_000
    d = synth.generate(n, seed=32)
    path = str(tmp_path / "t.bam")
    bamio.write_batch_bam(path, "chr1", n, d.batch)
    raw = bytearray(open(path, "rb").read())
    blocks = tp._file_blocks(path)
    off, size = blocks[-4]
    raw[off + size // 2] ^= 0x5a
    bad = str(tmp_path / "late.bam")
    open(bad, "wb").write(bytes(raw))
    os.link(path + ".bai", bad + ".bai")
    nb = bamdec.NativeBam(bad, threads=1)
    assert nb.plan("chr1", 0, 40_000).comp_bytes < len(raw) // 3
    _same_as_host(ctx, nb, "chr1", 0, 40_000)
    nb.close()


def _rewrite(raw, out):
    """the inflated stream -> BGZF blocks without a BAI (the rewrite of test_malformed_records_are_rejected_not_read_past)"""
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


def test_device_malformed_records_match_the_host(ctx, tmp_path):
    path = str(tmp_path / "ok.bam")
    tb._write(path, [tb._rec(pos=10, qname="first"), tb._rec(pos=20, qname="second")])
    raw = bytearray(gzip.open(path, "rb").read())
    first = raw.find(b"first\x00") - 36
    bs = struct.unpack_from("<I", raw, first)[0]
    rng = np.random.default_rng(5)
    muts = []
    m = bytearray(raw); struct.pack_into("<i", m, first + 4 + 16, 1 << 20); muts.append(m)
    m = bytearray(raw); m[first + 4 + 8] = 255; muts.append(m)
    m = bytearray(raw); struct.pack_into("<H", m, first + 4 + 12, 60000); muts.append(m)
    m = bytearray(raw); struct.pack_into("<I", m, first, 16); muts.append(m)
    m = bytearray(raw); m[first + 4 + bs - 1] = 65; muts.append(m)
    for _ in range(40):
        m = bytearray(raw)
        for _ in range(3):
            m[first + 4 + int(rng.integers(0, bs))] = int(rng.integers(0, 256))
        muts.append(m)
    n_rejected = 0
    for i, m in enumerate(muts):
        p = _rewrite(m, str(tmp_path / ("mut%d.bam" % i)))
        try:
            nb = bamdec.NativeBam(p, threads=1)
        except IOError:
            continue
        try:
            want = nb.read_batch("chr1", 0, 1000, seq=False)
        except pack.BatchFormatError as ex:
            nb.close()
            assert _device_error(ctx, p) == str(ex), i
            n_rejected += 1
            continue
        try:
            got = _device_batch(ctx, nb, "chr1", 0, 1000)
        except lib.HimutError as ex:  # the upload's checks reject the host decoder's batch with the same words
            with pytest.raises(lib.HimutError) as ex_host:
                ctx.upload(want)
            assert str(ex) == str(ex_host.value), i
            nb.close()
            continue
        for name in ("tstart", "tend", "qstart", "qlen", "mapq", "qname_id", "bq_off", "op_off", "n_ops", "bq", "ops"):
            assert np.array_equal(getattr(got, name), getattr(want, name)), (i, name)
        nb.close()
    assert n_rejected >= 5


def test_device_corrupt_block_and_bad_index(ctx, tmp_path):
    d = synth.generate(200_000, seed=31)
    path = str(tmp_path / "t.bam")
    bamio.write_batch_bam(path, "chr1", 200_000, d.batch)
    raw = bytearray(open(path, "rb").read())
    # a compressed byte in the middle of the file: the block fails to inflate or its CRC32
    bad = str(tmp_path / "crc.bam")
    m = bytearray(raw)
    blocks = tp._file_blocks(path)
    off, size = blocks[len(blocks) // 2]
    m[off + size // 2] ^= 0x5a  # inside the payload of a block in the middle
    open(bad, "wb").write(bytes(m))
    os.link(path + ".bai", bad + ".bai")
    msg = _device_error(ctx, bad, 0, 200_000)
    assert ("fails its CRC32" in msg or "does not inflate" in msg), msg
    # a BAI linear-index entry moved one byte into a record
    bai = bytearray(open(path + ".bai", "rb").read())
    q = 8 + 4
    nbin = struct.unpack_from("<i", bai, 8)[0]
    for _ in range(nbin):
        nchunk = struct.unpack_from("<i", bai, q + 4)[0]
        q += 8 + 16 * nchunk
    nintv = struct.unpack_from("<i", bai, q)[0]
    assert nintv > 4
    k = q + 4 + 8 * 3  # the fourth window's entry
    v = struct.unpack_from("<Q", bai, k)[0]
    struct.pack_into("<Q", bai, k, v + 1)
    moved = str(tmp_path / "moved.bam")
    os.link(path, moved)
    open(moved + ".bai", "wb").write(bytes(bai))
    msg = _device_error(ctx, moved, 0, 200_000)
    assert msg.startswith("BAI does not point at record starts"), msg


def _run_call_device(c, tmp_path, monkeypatch):
    seen = []
    orig = lib.Context.decode_region

    def spy(self, *a, **k):
        r = orig(self, *a, **k)
        seen.append({n for n, _ in self.last_decode_times})
        return r

    real = caller.call_region
    monkeypatch.setattr(lib.Context, "decode_region", spy)
    monkeypatch.setattr(caller, "call_region", lambda *a, **k: real(*a, **dict(k, decode="device")))
    out = tw._run_call(c, tmp_path)
    assert seen and any(DECODE_KERNELS <= s for s in seen)
    return out


@pytest.mark.parametrize("name", ["call_basic", "call_sets", "call_phase", "call_phase_indel", "call_adversarial_b"])
def test_call_worker_device_decode_matches_reference(name, tmp_path, monkeypatch):
    c = cases.build_case(name)
    fx = parity.load_golden(name)
    rows, log = _run_call_device(c, tmp_path, monkeypatch)
    gold = parity.golden_rows(fx)
    assert parity.rows_equal(rows, gold), parity.first_diff(rows, gold)
    assert log == fx["expected"]["log"]


def test_call_worker_device_decode_group_carry(tmp_path, monkeypatch):
    monkeypatch.setattr(worker, "GROUP_SPAN", 1200)
    for name in ("call_adversarial_a", "call_adversarial_b"):
        c = cases.build_case(name)
        fx = parity.load_golden(name)
        rows, log = _run_call_device(c, tmp_path, monkeypatch)
        gold = parity.golden_rows(fx)
        assert parity.rows_equal(rows, gold), parity.first_diff(rows, gold)
        assert log == fx["expected"]["log"]
