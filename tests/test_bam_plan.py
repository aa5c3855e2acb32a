"""Host plan of a region for the device decoder (hm_bam_region_plan): the compressed blocks and the record starts the
BAI gives, checked with Python's zlib against the file and against the host decoder's batch.  CPU only."""
import os
import struct
import zlib

import numpy as np
import pytest

import test_bamdec as tb
from himut_b200 import bamdec, bamio, synth


def _plan(nb, chrom, s, e):
    import ctypes as C
    p = nb.plan(chrom, s, e)
    n = int(p.n_blocks)
    get = lambda name, k, ct: np.array(C.cast(getattr(p, name), C.POINTER(ct))[:k]) if k and n else np.zeros(0)
    comp = C.string_at(p.comp, int(p.comp_bytes)) if p.comp_bytes else b""
    return dict(comp=comp, coff=get("blk_coff", n + 1, C.c_uint64), csize=get("blk_csize", n, C.c_uint32),
                isize=get("blk_isize", n, C.c_uint32), uoff=get("blk_uoff", n + 1, C.c_uint64), crc=get("blk_crc", n, C.c_uint32),
                entry=get("entry", int(p.n_entry), C.c_uint64), walk_end=int(p.walk_end), n_blocks=n)


def _inflate(pl):
    out = []
    for i in range(pl["n_blocks"]):
        o, cs = int(pl["coff"][i]), int(pl["csize"][i])
        blk = pl["comp"][o:o + cs]
        xlen = struct.unpack_from("<H", blk, 10)[0]
        data = zlib.decompress(blk[12 + xlen:cs - 8], -15)
        assert len(data) == pl["isize"][i] == struct.unpack_from("<I", blk, cs - 4)[0]
        assert zlib.crc32(data) & 0xffffffff == pl["crc"][i]
        assert sum(len(x) for x in out) == pl["uoff"][i]
        out.append(data)
    return b"".join(out)


def _file_blocks(path):
    """(offset, size) of every BGZF block of the file, by its own header walk"""
    raw = open(path, "rb").read()
    res, off = [], 0
    while off < len(raw):
        xlen = struct.unpack_from("<H", raw, off + 10)[0]
        bsize = None
        q = 0
        while q + 4 <= xlen:
            si, sl = raw[off + 12 + q:off + 14 + q], struct.unpack_from("<H", raw, off + 14 + q)[0]
            if si == b"BC":
                bsize = struct.unpack_from("<H", raw, off + 16 + q)[0]
            q += 4 + sl
        res.append((off, bsize + 1))
        off += bsize + 1
    return res


def _check(path, nb, chrom, s, e):
    pl = _plan(nb, chrom, s, e)
    host = nb.read_batch(chrom, s, e, seq=False)
    if pl["n_blocks"] == 0 or len(pl["entry"]) == 0:
        assert host.n_reads == 0
        return
    # the block table agrees with the file: the range is a run of its whole blocks, byte for byte
    raw = open(path, "rb").read()
    blocks = _file_blocks(path)
    base = raw.find(pl["comp"])
    k0 = [o for o, _c in blocks].index(base)
    assert [(o - base, c) for o, c in blocks[k0:k0 + pl["n_blocks"]]] == [(int(pl["coff"][i]), int(pl["csize"][i])) for i in range(pl["n_blocks"])]
    u = _inflate(pl)
    assert pl["walk_end"] <= len(u)
    # walk from the first entry: every entry point is a record start, and the range holds every record the host returns
    recs, p = {}, int(pl["entry"][0])
    while p + 4 <= pl["walk_end"]:
        bs = struct.unpack_from("<I", u, p)[0]
        if p + 4 + bs > pl["walk_end"]:
            break
        l_name = u[p + 4 + 8]
        name = u[p + 4 + 32:p + 4 + 32 + l_name - 1].decode()
        recs[p] = (name, struct.unpack_from("<i", u, p + 8)[0])
        p += 4 + bs
    assert set(int(x) for x in pl["entry"]) <= set(recs)
    have = set(recs.values())
    for r in range(host.n_reads):
        assert (nb.qname(int(host.qname_id[r])), int(host.tstart[r])) in have


def _write(path, parts, writer, level):
    if writer == "native":
        assert len(parts) == 1
        bamdec.write_batch_bam(path, parts[0][0], parts[0][1], parts[0][2], level=level)
    else:
        w = bamio.BamWriter(path, [(c, n) for c, n, _ in parts], level=level)
        for rid, (_c, _n, b) in enumerate(parts):
            bamio._add_batch(w, rid, b)
        w.close()


@pytest.mark.parametrize("writer", ["python", "native"])
@pytest.mark.parametrize("level", [1, 6])
def test_plan_of_random_regions(tmp_path, writer, level):
    n = 150_000
    d = synth.generate(n, seed=21)
    path = str(tmp_path / "p.bam")
    _write(path, [("chr1", n, d.batch)], writer, level)
    nb = bamdec.NativeBam(path, threads=2)
    rng = np.random.default_rng(level)
    regions = [(0, n), (0, 1), (n - 1, n), (70_000, 70_001), (n + 10, n + 500), (n - 100, n + 100)]
    for _ in range(8):
        s = int(rng.integers(0, n))
        regions.append((s, s + int(rng.integers(1, 40_000))))
    for s, e in regions:
        _check(path, nb, "chr1", s, e)
    nb.close()


@pytest.mark.parametrize("level", [1, 6])
def test_plan_multi_contig_and_empty_contig(tmp_path, level):
    a, b = synth.generate(60_000, seed=22), synth.generate(40_000, seed=23)
    empty = synth.generate(20_000, seed=24).batch.select(np.zeros(0, np.int64))
    path = str(tmp_path / "m.bam")
    _write(path, [("chr1", 60_000, a.batch), ("chrE", 20_000, empty), ("chr2", 40_000, b.batch)], "python", level)
    nb = bamdec.NativeBam(path, threads=2)
    for chrom, n in (("chr1", 60_000), ("chrE", 20_000), ("chr2", 40_000)):
        for s, e in ((0, n), (0, 1), (n - 1, n), (n // 2, n // 2 + 5000), (n + 5, n + 50)):
            _check(path, nb, chrom, s, e)
    assert len(_plan(nb, "chrE", 0, 20_000)["entry"]) == 0
    nb.close()


def test_plan_without_index_is_the_whole_file(tmp_path):
    d = synth.generate(60_000, seed=13)
    path = str(tmp_path / "t.bam")
    bamio.write_batch_bam(path, "chr1", 60_000, d.batch)
    os.remove(path + ".bai")
    nb = bamdec.NativeBam(path, threads=2)
    assert not nb.has_index
    pl = _plan(nb, "chr1", 20_000, 30_000)
    assert len(pl["entry"]) == 1 and pl["walk_end"] == len(_inflate(pl))
    _check(path, nb, "chr1", 20_000, 30_000)
    nb.close()


def test_plan_of_a_small_hand_written_bam(tmp_path):
    path = str(tmp_path / "m.bam")
    tb._write(path, [tb._rec(pos=10, qname="a"), tb._rec(pos=400, qname="b"), tb._rec(pos=5, ref_id=1, qname="c")])
    nb = bamdec.NativeBam(path, threads=1)
    for chrom in ("chr1", "chr2"):
        for s, e in ((0, 1000), (15, 16), (0, 11), (500, 2000)):
            _check(path, nb, chrom, s, e)
    nb.close()


def test_intern_qnames_gives_the_host_decoders_ids(tmp_path):
    d = synth.generate(60_000, seed=25)
    path = str(tmp_path / "t.bam")
    bamio.write_batch_bam(path, "chr1", 60_000, d.batch)
    nb = bamdec.NativeBam(path, threads=1)
    first = nb.read_batch("chr1", 0, 30_000, seq=False)
    names = [nb.qname(int(i)) for i in first.qname_id]
    later = nb.read_batch("chr1", 25_000, 60_000, seq=False)
    want = later.qname_id.copy()
    blob = b"".join(n.encode() + b"\0" for n in [nb.qname(int(i)) for i in want])
    off = np.cumsum([0] + [len(nb.qname(int(i))) + 1 for i in want])[:-1].astype(np.uint64)
    buf = np.frombuffer(blob, np.uint8).copy()
    got = nb.intern_qnames(buf, off, len(want))
    assert np.array_equal(got, want)
    # names never seen before get the next ids, as the host decoder would give them
    n0 = nb.n_qnames()
    new = np.frombuffer(b"zz1\0zz2\0zz1\0", np.uint8).copy()
    assert nb.intern_qnames(new, np.array([0, 4, 8], np.uint64), 3).tolist() == [n0, n0 + 1, n0]
    assert names and nb.qname(n0) == "zz1"
    nb.close()
