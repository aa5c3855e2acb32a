"""BAMs indexed with a CSI: the index lookup (<bam>.bai, <bam>.csi, <stem>.bai, <stem>.csi), the CSI parser and its
rejections, index-driven fetch in the Python specification (bamio) and the native host decoder against a scan from the
first record, the device decoder's plan under a CSI against the plan under a BAI, and the two writers' CSIs against
each other.  CPU only."""
import gzip
import os
import shutil
import struct
import zlib

import numpy as np
import pytest

import test_bam_plan as tp
import test_bamdec as tb
from himut_b200 import bamdec, bamio, bamlib, pack, synth

PARAMS = [(14, 5), (12, 6), (16, 4)]
LONG = 2**31 - 1


def _write(path, parts, writer, **index):
    if writer == "native":
        assert len(parts) == 1
        bamdec.write_batch_bam(path, parts[0][0], parts[0][1], parts[0][2], **index)
    else:
        bamio.write_batches_bam(path, parts, **index)


def _same(x, name_x, y, name_y):
    """the same batch; query-name ids are interned per handle, so they are compared as the names they stand for"""
    for name, _ in x._FIELDS:
        a, b = getattr(x, name), getattr(y, name)
        if name == "qname_id":
            a, b = np.array([name_x(int(i)) for i in a]), np.array([name_y(int(i)) for i in b])
        assert a.shape == b.shape and np.array_equal(a, b), name


def _scan_copy(path, tmp_path):
    """the same BAM under a name no index goes with: every fetch scans from the first record"""
    bare = str(tmp_path / ("bare_%s" % os.path.basename(path)))
    shutil.copyfile(path, bare)
    return bare


# ---------------------------------------------------------------------------------------------------- CSI contents
def _block_table(path):
    """(file offset, offset in the inflated stream) of every BGZF block of a file"""
    raw = open(path, "rb").read()
    out, u = {}, 0
    for off, size in tp._file_blocks(path):
        out[off] = u
        u += struct.unpack_from("<I", raw, off + size - 4)[0]
    return out, u


def _record_starts(path):
    """inflated-stream offset -> ordinal of every record, and the end of the last one"""
    r = bamio.BamReader(path)
    blocks, _ = _block_table(path)
    r.bg.seek(r.first_record)
    starts, k = {}, 0
    while True:
        v = r.bg.tell()
        head = r.bg.read(4)
        if len(head) < 4:
            break
        starts[blocks[v >> 16] + (v & 0xFFFF)] = k
        r.bg.read(struct.unpack("<i", head)[0])
        k += 1
    r.close()
    return starts, k


def parse_csi(path):
    """-> (min_shift, depth, [ {bin: (loffset, [(beg, end), ...])} per reference ], n_no_coor): the file as written"""
    d = gzip.decompress(open(path, "rb").read())
    assert d[:4] == b"CSI\x01"
    ms, depth, l_aux = struct.unpack_from("<iii", d, 4)
    p = 16 + l_aux
    n_ref, = struct.unpack_from("<i", d, p)
    p += 4
    refs = []
    for _ in range(n_ref):
        n_bin, = struct.unpack_from("<i", d, p)
        p += 4
        bins = {}
        for _b in range(n_bin):
            b, loff, n = struct.unpack_from("<IQi", d, p)
            p += 16
            bins[b] = (loff, [struct.unpack_from("<QQ", d, p + 16 * c) for c in range(n)])
            p += 16 * n
        refs.append(bins)
    n_no_coor = struct.unpack_from("<Q", d, p)[0] if p + 8 <= len(d) else None
    return ms, depth, refs, n_no_coor


def _as_records(path, csi):
    """the CSI with every virtual offset replaced by the ordinal of the record it points at (n: the end of the last)"""
    blocks, _ = _block_table(path)
    starts, n = _record_starts(path)

    def rec(v, end=False):
        u = blocks.get(v >> 16, -1) + (v & 0xFFFF)
        assert u in starts or end, v
        return starts.get(u, n)
    ms, depth, refs, nnc = csi
    pseudo = bamio.pseudo_bin(depth)
    out = []
    for bins in refs:
        o = {}
        for b, (loff, chunks) in bins.items():
            if b == pseudo:
                o[b] = (rec(chunks[0][0]), rec(chunks[0][1], True), chunks[1][0])
            else:
                o[b] = (rec(loff), [(rec(x), rec(y, True)) for x, y in chunks])
        out.append(o)
    return ms, depth, out, nnc


def _shifted(batch, off):
    from himut_b200 import abi
    kw = {name: getattr(batch, name) for name, _ in abi.ReadBatch._FIELDS}
    kw["tstart"] = (batch.tstart.astype(np.int64) + off).astype(np.int32)
    kw["tend"] = (batch.tend.astype(np.int64) + off).astype(np.int32)
    return abi.ReadBatch(**kw)


@pytest.fixture(scope="module")
def d150():
    return synth.generate(150_000, seed=21)


@pytest.mark.parametrize("ms,depth", PARAMS + [(14, None)])
def test_python_and_native_csi_hold_the_same_bins(tmp_path, d150, ms, depth):
    """the two writers cut blocks differently, so offsets differ; read as the records they point at, every bin, chunk,
    loffset and the pseudo-bin agree.  depth None: htslib's default for a contig of 2^31 - 1 (reads near its end)"""
    n, batch = 150_000, d150.batch
    contig = n if depth else LONG
    if depth is None:
        batch = _shifted(batch, LONG - n - 10)
    got = {}
    for writer in ("python", "native"):
        path = str(tmp_path / ("%s.bam" % writer))
        _write(path, [("chr1", contig, batch)], writer, index="csi", min_shift=ms, depth=depth)
        assert os.path.exists(path + ".csi") and not os.path.exists(path + ".bai")
        csi = parse_csi(path + ".csi")
        assert csi[0] == ms and csi[1] == (depth or bamio.default_depth([contig], ms)) and csi[3] == 0
        got[writer] = _as_records(path, csi)
    assert got["python"] == got["native"]
    bins = got["native"][2][0]
    pseudo = bamio.pseudo_bin(got["native"][1])
    assert bins[pseudo] == (0, batch.n_reads, batch.n_reads)
    assert len(bins) > 3
    if depth is None:
        assert got["native"][1] == 6 and pseudo == 299_594  # 2^(14 + 18) >= 2^31 - 1 + 256


def test_default_depth_is_htslibs():
    assert bamio.default_depth([1000]) == 0 and bamio.default_depth([2**14 - 256]) == 0 and bamio.default_depth([2**14 - 255]) == 1
    assert bamio.default_depth([2**29 - 256]) == 5 and bamio.default_depth([2**29]) == 6 and bamio.default_depth([LONG]) == 6
    assert bamio.pseudo_bin(5) == 37450 and bamio.pseudo_bin(6) == 299594


def test_bai_is_refused_past_2_29(tmp_path, d150):
    with pytest.raises(ValueError):
        bamio.BamWriter(str(tmp_path / "x.bam"), [("chr1", 2**29 + 1)])
    with pytest.raises(ValueError):
        bamdec.write_batch_bam(str(tmp_path / "y.bam"), "chr1", 2**29 + 1, d150.batch)
    bamio.BamWriter(str(tmp_path / "z.bam"), [("chr1", 2**29)]).close()


def test_records_past_2_29_carry_a_bin_no_one_reads(tmp_path, d150):
    batch = _shifted(d150.batch, 2**30)
    for writer in ("python", "native"):
        path = str(tmp_path / ("%s.bam" % writer))
        _write(path, [("chr1", LONG, batch)], writer, index="csi")
        r = bamio.BamReader(path)
        r.bg.seek(r.first_record)
        size = struct.unpack("<i", r.bg.read(4))[0]
        assert struct.unpack_from("<H", r.bg.read(size), 10)[0] == 4680
        r.close()


# ---------------------------------------------------------------------------------------------------- fetch
def _regions(n):
    return [(0, n), (1, 2 * n // 3), (2 * n // 3, n - 2), (n // 2, n // 2 + 1), (n - 10, n), (0, 1), (n + 5, n + 50),
            (n // 3, n // 3), (n // 4, n // 4 - 100), (7_000, 70_000)]


def _all_agree(path, bare, chrom, n, off=0):
    nb, scan = bamdec.NativeBam(path, threads=2), bamdec.NativeBam(bare, threads=2)
    r, r_scan = bamio.BamReader(path), bamio.BamReader(bare)
    assert nb.index_kind == r.index_kind == "csi" and scan.index_kind == r_scan.index_kind == "none"
    total = 0
    for s, e in _regions(n):
        s, e = s + off, e + off
        want = scan.read_batch(chrom, s, e)
        _same(nb.read_batch(chrom, s, e), nb.qname, want, scan.qname)
        bb = pack.BatchBuilder()
        spec = bamio.read_batch(r, chrom, s, e, builder=bb)
        _same(spec, {v: k for k, v in bb.qnames.items()}.get, want, scan.qname)
        total += want.n_reads
    for s, e in ((off, off + n // 2), (off + n // 3, off + n)):
        assert list(nb.window_qlens(chrom, s, e)) == list(scan.window_qlens(chrom, s, e))
    for x in (nb, scan, r, r_scan):
        x.close()
    return total


@pytest.mark.parametrize("writer", ["python", "native"])
@pytest.mark.parametrize("ms,depth", PARAMS)
def test_index_fetch_equals_a_scan(tmp_path, d150, writer, ms, depth):
    n = 150_000
    path = str(tmp_path / "t.bam")
    _write(path, [("chr1", n, d150.batch)], writer, index="csi", min_shift=ms, depth=depth)
    assert _all_agree(path, _scan_copy(path, tmp_path), "chr1", n) > 0


@pytest.mark.parametrize("writer", ["python", "native"])
def test_index_fetch_on_a_contig_of_2_31(tmp_path, d150, writer):
    """reads in the last 200 kb of a contig of 2^31 - 1, at the writer's default depth"""
    n, off = 150_000, LONG - 150_000 - 1
    path = str(tmp_path / "t.bam")
    _write(path, [("chr1", LONG, _shifted(d150.batch, off))], writer, index="csi")
    assert _all_agree(path, _scan_copy(path, tmp_path), "chr1", n, off) > 0


def test_multi_contig_with_an_empty_contig(tmp_path):
    a, b = synth.generate(60_000, seed=22), synth.generate(40_000, seed=23)
    empty = synth.generate(20_000, seed=24).batch.select(np.zeros(0, np.int64))
    for ms, depth in PARAMS:
        path = str(tmp_path / ("m%d.bam" % ms))
        bamio.write_batches_bam(path, [("chr1", 60_000, a.batch), ("chrE", 20_000, empty), ("chr2", 40_000, b.batch)],
                                index="csi", min_shift=ms, depth=depth)
        bare = _scan_copy(path, tmp_path)
        for chrom, n in (("chr1", 60_000), ("chrE", 20_000), ("chr2", 40_000)):
            got = _all_agree(path, bare, chrom, n)
            assert (got == 0) == (chrom == "chrE")


def test_hand_written_records_and_csi(tmp_path):
    """secondary, supplementary and soft-clipped records on two contigs, through a CSI"""
    path = str(tmp_path / "m.bam")
    w = bamio.BamWriter(path, [("chr1", 1000), ("chr2", 1000)], index="csi", min_shift=4, depth=3)
    for r in [tb._rec(pos=10, qname="a"), tb._rec(pos=12, flag=0x100, qname="s", cs=None), tb._rec(pos=14, flag=0x800, qname="p"),
              tb._rec(pos=400, qname="b"), tb._rec(pos=5, ref_id=1, qname="c"), tb._rec(pos=900, ref_id=1, qname="d")]:
        w.add(**r)
    w.close()
    bare = _scan_copy(path, tmp_path)
    nb, scan = bamdec.NativeBam(path, threads=1), bamdec.NativeBam(bare, threads=1)
    for chrom in ("chr1", "chr2"):
        for s, e in ((0, 1000), (15, 16), (0, 11), (500, 2000), (17, 17), (899, 900)):
            _same(nb.read_batch(chrom, s, e), nb.qname, scan.read_batch(chrom, s, e), scan.qname)
            tp._check(path, nb, chrom, s, e)
    nb.close()
    scan.close()


# ---------------------------------------------------------------------------------------------------- lookup
def test_lookup_order_and_index_kind(tmp_path, d150):
    n = 150_000
    src = str(tmp_path / "src")
    os.makedirs(src)
    bamdec.write_batch_bam(os.path.join(src, "x.bam"), "chr1", n, d150.batch)
    bamdec.write_batch_bam(os.path.join(src, "y.bam"), "chr1", n, d150.batch, index="csi")
    bam = open(os.path.join(src, "x.bam"), "rb").read()
    assert bam == open(os.path.join(src, "y.bam"), "rb").read()  # the index does not change the BAM
    bai, csi = os.path.join(src, "x.bam.bai"), os.path.join(src, "y.bam.csi")
    layouts = {"x.bam.bai": ("bai", [("x.bam.bai", bai)]), "x.bai": ("bai", [("x.bai", bai)]),
               "x.bam.csi": ("csi", [("x.bam.csi", csi)]), "x.csi": ("csi", [("x.csi", csi)]),
               "both": ("bai", [("x.bam.bai", bai), ("x.bam.csi", csi)]), "stem bai, bam csi": ("csi", [("x.bai", bai), ("x.bam.csi", csi)]),
               "none": ("none", [])}
    batches, names = [], []
    for name, (kind, files) in layouts.items():
        d = tmp_path / name.replace(" ", "_").replace(",", "")
        os.makedirs(d)
        path = str(d / "x.bam")
        open(path, "wb").write(bam)
        for f, srcf in files:
            shutil.copyfile(srcf, str(d / f))
        nb = bamdec.NativeBam(path, threads=2)
        r = bamio.BamReader(path)
        assert nb.index_kind == r.index_kind == kind, name
        assert nb.has_index == (nb.lib.hm_bam_index_kind(nb.h) != 0) == (kind != "none")
        batches.append(nb.read_batch("chr1", 40_000, 90_000))
        bb = pack.BatchBuilder()
        spec = bamio.read_batch(r, "chr1", 40_000, 90_000, builder=bb)
        _same(spec, {v: k for k, v in bb.qnames.items()}.get, batches[-1], nb.qname)
        names.append({int(i): nb.qname(int(i)) for i in batches[-1].qname_id})
        nb.close()
        r.close()
    for b, nm in zip(batches[1:], names[1:]):
        _same(b, nm.get, batches[0], names[0].get)
    assert batches[0].n_reads > 0


# ---------------------------------------------------------------------------------------------------- rejections
def _csi_bytes(path):
    return gzip.decompress(open(path + ".csi", "rb").read())


def _put(tmp_path, bam, name, payload, raw=False):
    path = str(tmp_path / name)
    os.link(bam, path)
    open(path + ".csi", "wb").write(payload if raw else bamio._bgzf_block(payload, 1) + bamio._BGZF_EOF)
    return path


def _rejected(path, *what):
    with pytest.raises(IOError) as ex:
        bamdec.NativeBam(path)
    msg = str(ex.value)
    assert path + ".csi" in msg.split("as BAM: ", 1)[-1], msg
    for w in what:
        assert w in msg, msg
    with pytest.raises(bamio.BamError) as ex:
        bamio.BamReader(path)
    assert path + ".csi" in str(ex.value)


def _fields(d):
    """(offset, name) of every field of a single-reference CSI, in file order"""
    ms, depth, l_aux = struct.unpack_from("<iii", d, 4)
    out = [(0, "magic"), (4, "min_shift"), (8, "depth"), (12, "l_aux")]
    p = 16 + l_aux
    out.append((p, "n_ref"))
    p += 4
    out.append((p, "n_bin"))
    n_bin, = struct.unpack_from("<i", d, p)
    p += 4
    for _ in range(n_bin):
        b, _l, n = struct.unpack_from("<IQi", d, p)
        out += [(p, "bin %d" % b), (p + 4, "loffset"), (p + 12, "n_chunk")]
        p += 16
        for c in range(n):
            out += [(p, "chunk_beg"), (p + 8, "chunk_end")]
            p += 16
    out.append((p, "n_no_coor"))
    return out


def test_corrupt_csi_files_are_rejected_with_the_file_named(tmp_path, d150):
    n = 150_000
    bam = str(tmp_path / "t.bam")
    bamdec.write_batch_bam(bam, "chr1", n, d150.batch, index="csi", min_shift=14, depth=5)
    d = _csi_bytes(bam)
    fields = _fields(d)
    _rejected(_put(tmp_path, bam, "magic.bam", b"CSJ\x01" + d[4:]), "not a CSI index")
    _rejected(_put(tmp_path, bam, "plain.bam", d, raw=True), "not a BGZF-compressed CSI index")
    _rejected(_put(tmp_path, bam, "gzip.bam", gzip.compress(d), raw=True), "not a BGZF-compressed CSI index")
    _rejected(_put(tmp_path, bam, "empty.bam", b"", raw=True), "not a CSI index")
    # a compressed CSI cut short, and one whose CRC does not match
    z = open(bam + ".csi", "rb").read()
    _rejected(_put(tmp_path, bam, "cut.bam", z[:len(z) // 2], raw=True), "not a BGZF-compressed CSI index")
    flip = bytearray(z)
    flip[len(z) - 28 - 8] ^= 1
    _rejected(_put(tmp_path, bam, "crc.bam", bytes(flip), raw=True), "not a BGZF-compressed CSI index")
    # the span of the scheme shorter than the contig: min_shift 14 and depth 2 cover 1 Mb
    _rejected(_put(tmp_path, bam, "span.bam", d[:8] + struct.pack("<i", 0) + d[12:]), "cover 16384 positions, chr1 has 150000")
    _rejected(_put(tmp_path, bam, "depth.bam", d[:8] + struct.pack("<i", 11) + d[12:]), "unsupported min_shift")
    _rejected(_put(tmp_path, bam, "laux.bam", d[:12] + struct.pack("<i", len(d)) + d[16:]), "l_aux")
    _rejected(_put(tmp_path, bam, "laux_neg.bam", d[:12] + struct.pack("<i", -1) + d[16:]), "l_aux")
    nbin_at = next(o for o, f in fields if f == "n_bin")
    _rejected(_put(tmp_path, bam, "nbin.bam", d[:nbin_at] + struct.pack("<i", 1 << 28) + d[nbin_at + 4:]), "n_bin")
    _rejected(_put(tmp_path, bam, "nbin_neg.bam", d[:nbin_at] + struct.pack("<i", -2) + d[nbin_at + 4:]), "n_bin")
    bin_at = next(o for o, f in fields if f.startswith("bin "))
    _rejected(_put(tmp_path, bam, "bin.bam", d[:bin_at] + struct.pack("<I", 37451) + d[bin_at + 4:]), "bin 37451 past the pseudo-bin 37450")
    _rejected(_put(tmp_path, bam, "bin_last.bam", d[:bin_at] + struct.pack("<I", 37449) + d[bin_at + 4:]), "bin 37449 past the pseudo-bin 37450")
    nch_at = next(o for o, f in fields if f == "n_chunk")
    _rejected(_put(tmp_path, bam, "nchunk.bam", d[:nch_at] + struct.pack("<i", 1 << 27) + d[nch_at + 4:]), "n_chunk")
    _rejected(_put(tmp_path, bam, "nchunk_neg.bam", d[:nch_at] + struct.pack("<i", -1) + d[nch_at + 4:]), "n_chunk")
    beg_at = next(o for o, f in fields if f == "chunk_beg")
    end = struct.unpack_from("<Q", d, beg_at + 8)[0]
    _rejected(_put(tmp_path, bam, "chunk.bam", d[:beg_at] + struct.pack("<Q", end + 1) + d[beg_at + 8:]), "begins after its end")
    # truncation inside every field (n_no_coor is optional: a file cut before it is whole)
    for k, (o, f) in enumerate(fields[:-1]):
        cut = o + 1 if f != "magic" else 2
        _rejected(_put(tmp_path, bam, "trunc%d.bam" % k, d[:cut]))
    # what is intact still opens: n_no_coor left out, and the file as written
    nb = bamdec.NativeBam(_put(tmp_path, bam, "no_nnc.bam", d[:fields[-1][0]]))
    assert nb.index_kind == "csi" and nb.read_batch("chr1", 0, n).n_reads == d150.batch.n_reads
    nb.close()


# ---------------------------------------------------------------------------------------------------- plans
def _abs_plan(path, nb, chrom, s, e):
    """the plan with its range and entry points as offsets in the file's whole inflated stream"""
    pl = tp._plan(nb, chrom, s, e)
    if pl["n_blocks"] == 0:
        return pl, None
    raw = open(path, "rb").read()
    blocks, _ = _block_table(path)
    base = raw.find(pl["comp"])
    u0 = blocks[base]
    return pl, dict(start=u0 + int(pl["entry"][0]) if len(pl["entry"]) else None, walk_end=u0 + pl["walk_end"],
                    last_block=base + int(pl["coff"][pl["n_blocks"]]), entries=[u0 + int(x) for x in pl["entry"]])


@pytest.mark.parametrize("writer", ["python", "native"])
def test_csi_plan_ends_where_the_bai_plan_ends(tmp_path, d150, writer):
    n = 150_000
    bai, csi = str(tmp_path / "b.bam"), str(tmp_path / "c.bam")
    _write(bai, [("chr1", n, d150.batch)], writer)
    _write(csi, [("chr1", n, d150.batch)], writer, index="csi", min_shift=14, depth=5)
    assert open(bai, "rb").read() == open(csi, "rb").read()
    nb_b, nb_c = bamdec.NativeBam(bai, threads=2), bamdec.NativeBam(csi, threads=2)
    rng = np.random.default_rng(5)
    regions = _regions(n) + [(int(s), int(s) + int(rng.integers(1, 40_000))) for s in rng.integers(0, n, 12)]
    for s, e in regions:
        pb, ab = _abs_plan(bai, nb_b, "chr1", s, e)
        pc, ac = _abs_plan(csi, nb_c, "chr1", s, e)
        tp._check(csi, nb_c, "chr1", s, e)
        assert (ab is None) == (ac is None), (s, e)
        if ab is None or ab["start"] is None:
            continue
        assert ac["walk_end"] == ab["walk_end"] and ac["last_block"] == ab["last_block"], (s, e)
        assert ac["start"] <= ab["start"], (s, e)
    nb_b.close()
    nb_c.close()


@pytest.mark.parametrize("ms,depth", PARAMS)
def test_csi_plans_at_every_depth(tmp_path, d150, ms, depth):
    n = 150_000
    for writer in ("python", "native"):
        path = str(tmp_path / ("%s.bam" % writer))
        _write(path, [("chr1", n, d150.batch)], writer, index="csi", min_shift=ms, depth=depth, level=6)
        nb = bamdec.NativeBam(path, threads=2)
        for s, e in _regions(n):
            tp._check(path, nb, "chr1", s, e)
        nb.close()


def test_plans_of_the_64mb_contig_groups(tmp_path, capsys):
    """the contig of tools/worker_trace.py (64 Mb, 30x, seed 5) under a BAI and under a CSI of (14, 5): for each of
    its four 16 Mb decode groups the same compressed range, and the entry points each index gives k_bam_walk"""
    n = 64_000_000
    d = synth.generate(n, seed=5, copy=False)
    bai, csi = str(tmp_path / "b.bam"), str(tmp_path / "c.bam")
    bamdec.write_batch_bam(bai, "chr1", n, d.batch)
    bamdec.write_batch_bam(csi, "chr1", n, d.batch, index="csi", min_shift=14, depth=5)
    del d
    assert os.path.getsize(bai) == os.path.getsize(csi)
    nb_b, nb_c = bamdec.NativeBam(bai), bamdec.NativeBam(csi)
    rows = []
    for g in range(0, n, 16_000_000):
        pb, pc = tp._plan(nb_b, "chr1", g, g + 16_000_000), tp._plan(nb_c, "chr1", g, g + 16_000_000)
        # one compressed range: the same first entry point, blocks and walk end (the file bytes are the same)
        assert len(pb["comp"]) == len(pc["comp"]) and pb["comp"][:4096] == pc["comp"][:4096]
        assert pb["entry"][0] == pc["entry"][0] and pb["walk_end"] == pc["walk_end"] and pb["n_blocks"] == pc["n_blocks"]
        assert np.array_equal(pb["coff"], pc["coff"])
        assert len(pc["entry"]) > 0
        rows.append((g, len(pb["comp"]), len(pb["entry"]), len(pc["comp"]), len(pc["entry"])))
    with capsys.disabled():
        print("\n16 Mb group: BAI compressed bytes, entry points | CSI (14, 5) compressed bytes, entry points")
        for r in rows:
            print("  %9d: %11d %6d | %11d %6d" % r)
    nb_b.close()
    nb_c.close()


# ---------------------------------------------------------------------------------------------------- pre-pass
def test_thresholds_through_a_csi(tmp_path):
    """bamlib.get_thresholds (the BAM pre-pass, 100 windows per contig) gives the same thresholds through a CSI as
    through the BAI of the same BAM"""
    parts = [("chr1", 300_000, synth.generate(300_000, seed=61).batch), ("chr2", 200_000, synth.generate(200_000, seed=62).batch)]
    bai, csi = str(tmp_path / "b.bam"), str(tmp_path / "c.bam")
    bamio.write_batches_bam(bai, parts)
    bamio.write_batches_bam(csi, parts, index="csi", min_shift=12, depth=6)
    chroms, lens = [c for c, _, _ in parts], {c: n for c, n, _ in parts}
    assert bamdec.NativeBam(csi).index_kind == "csi"
    assert bamlib.get_thresholds(csi, chroms, lens) == bamlib.get_thresholds(bai, chroms, lens)


def test_offsets_past_the_end_of_the_bam_are_rejected(tmp_path, d150):
    """an loffset or a chunk past the end of the BAM would read as an empty region: refused at open"""
    n = 150_000
    bam = str(tmp_path / "t.bam")
    bamdec.write_batch_bam(bam, "chr1", n, d150.batch, index="csi", min_shift=14, depth=5)
    d = _csi_bytes(bam)
    far = (os.path.getsize(bam) + 100) << 16
    for what in ("loffset", "chunk_beg"):
        m = bytearray(d)
        o = [o for o, f in _fields(d) if f == what][0]
        struct.pack_into("<Q", m, o, far)
        if what == "chunk_beg":
            struct.pack_into("<Q", m, o + 8, far)
        _rejected(_put(tmp_path, bam, "far_%s.bam" % what, bytes(m)), "points past the end of the BAM")


def test_zlib_reads_what_the_writers_compress(tmp_path, d150):
    for writer in ("python", "native"):
        path = str(tmp_path / ("%s.bam" % writer))
        _write(path, [("chr1", 150_000, d150.batch)], writer, index="csi")
        raw = open(path + ".csi", "rb").read()
        assert raw.endswith(bamio._BGZF_EOF)
        for off, size in tp._file_blocks(path + ".csi"):
            blk = raw[off:off + size]
            xlen = struct.unpack_from("<H", blk, 10)[0]
            data = zlib.decompress(blk[12 + xlen:size - 8], -15)
            assert zlib.crc32(data) == struct.unpack_from("<I", blk, size - 8)[0]
