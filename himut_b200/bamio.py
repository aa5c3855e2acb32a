"""Minimal BAM / BGZF / BAI / CSI reader and writer (pure Python + zlib).

pysam / htslib are not available in this image (SURVEY.md §0.4), and the worker mirrors need the
records of a region as a packed ReadBatch rather than as Python objects anyway.  The reader
implements what the reference touches through pysam (SURVEY.md §8b): header text, @SQ table,
fetch(chrom, start, end) — records overlapping the 0-based half-open window, in file order,
secondary / supplementary included — and the per-record fields reference_start/end,
query_alignment_start/end, query_sequence, query_qualities, mapping_quality, flag, cs:Z, tp:A, and
beyond it the CIGAR and MD:Z (records without cs:Z are decoded from CIGAR + MD, pack.parse_md, and records with
neither tag from CIGAR + the contig's reference sequence when the caller gives it, pack.parse_ref).
The reader seeks with the first index it finds of <bam>.bai, <bam>.csi, <stem>.bai and <stem>.csi (the names htslib
finds).  The writer exists for tests and for the synthetic-data tools (coordinate-sorted BAM + .bai or .csi).
"""
import io
import os
import struct
import zlib

import numpy as np

from . import abi, pack

_SEQ_DEC = "=ACMGRSVTWYHKDBN"
# BAM 4-bit base code -> our 2-bit code (A0 T1 G2 C3), 255 = not A/C/G/T
_NIB2CODE = np.full(16, 255, np.uint8)
_NIB2CODE[1], _NIB2CODE[2], _NIB2CODE[4], _NIB2CODE[8] = 0, 3, 2, 1
_CIGAR_REF = (1, 0, 1, 1, 0, 0, 0, 1, 1)    # M I D N S H P = X consume reference?
_CIGAR_QRY = (1, 1, 0, 0, 1, 0, 0, 1, 1)    # ... consume query?
_BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


BAI_MAX_LEN = 1 << 29  # the BAI binning scheme ends there: a longer contig can only be indexed with a CSI


class BamError(IOError):
    pass


# ------------------------------------------------------------------------------ BGZF
def _read_block(f):
    """-> (compressed size, payload bytes) of the BGZF block at the file position, or (0, b"")"""
    head = f.read(18)
    if len(head) == 0:
        return 0, b""
    if len(head) < 18 or head[:4] != b"\x1f\x8b\x08\x04":
        raise BamError("not a BGZF block")
    xlen = struct.unpack_from("<H", head, 10)[0]
    extra = head[12:18] + f.read(xlen - 6)
    bsize, p = None, 0
    while p + 4 <= len(extra):
        si1, si2, slen = extra[p], extra[p + 1], struct.unpack_from("<H", extra, p + 2)[0]
        if si1 == 66 and si2 == 67:
            bsize = struct.unpack_from("<H", extra, p + 4)[0]
        p += 4 + slen
    if bsize is None:
        raise BamError("BGZF block without BC field")
    rest = f.read(bsize + 1 - 12 - xlen)
    data = zlib.decompress(rest[:-8], -15)
    return bsize + 1, data


class _BgzfReader:
    def __init__(self, path):
        self.f = open(path, "rb")
        self.block_off = 0
        self.buf = b""
        self.pos = 0
        self.next_off = 0

    def seek(self, voffset):
        coff, uoff = voffset >> 16, voffset & 0xFFFF
        self.f.seek(coff)
        self.block_off = coff
        n, self.buf = _read_block(self.f)
        self.next_off = coff + n
        self.pos = uoff

    def tell(self):
        return (self.block_off << 16) | self.pos

    def read(self, n):
        out = []
        while n > 0:
            if self.pos >= len(self.buf):
                self.block_off = self.next_off
                self.f.seek(self.block_off)
                size, self.buf = _read_block(self.f)
                self.pos = 0
                if size == 0:
                    break
                self.next_off = self.block_off + size
                continue
            take = min(n, len(self.buf) - self.pos)
            out.append(self.buf[self.pos:self.pos + take])
            self.pos += take
            n -= take
        return b"".join(out)

    def close(self):
        self.f.close()


class Record:
    """decoded alignment (attribute names follow pysam.AlignedSegment)"""
    __slots__ = ("ref_id", "reference_start", "reference_end", "query_name", "flag", "mapping_quality",
                 "query_alignment_start", "query_alignment_end", "seq_nibbles", "l_seq", "qual", "tags",
                 "hard_clipped", "cigar")

    @property
    def is_secondary(self):
        return bool(self.flag & 0x100)

    @property
    def is_supplementary(self):
        return bool(self.flag & 0x800)

    @property
    def query_sequence(self):
        nb = np.frombuffer(self.seq_nibbles, dtype=np.uint8)
        codes = np.empty(nb.size * 2, np.uint8)
        codes[0::2], codes[1::2] = nb >> 4, nb & 15
        return "".join(_SEQ_DEC[c] for c in codes[: self.l_seq])

    @property
    def query_qualities(self):
        import array
        if self.l_seq and self.qual[0] == 0xFF:
            return None
        return array.array("B", self.qual)

    def get_tag(self, t):
        return self.tags[t]

    def has_tag(self, t):
        return t in self.tags


_B_SIZE = {"c": 1, "C": 1, "s": 2, "S": 2, "i": 4, "I": 4, "f": 4}
_TAG_FMT = {"c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I", "f": "f"}


def _parse_tags(buf, p, end, want=("cs", "tp", "MD")):
    tags = {}
    while p < end:
        tag = buf[p:p + 2].decode()
        ty = chr(buf[p + 2])
        p += 3
        if ty == "Z" or ty == "H":
            q = buf.index(b"\0", p)
            if tag in want:
                tags[tag] = buf[p:q].decode()
            p = q + 1
        elif ty == "A":
            if tag in want:
                tags[tag] = chr(buf[p])
            p += 1
        elif ty in "cC":
            p += 1
        elif ty in "sS":
            p += 2
        elif ty in "iIf":
            p += 4
        elif ty == "B":
            sub = chr(buf[p])
            if sub not in _B_SIZE:  # htslib rejects the record too
                raise BamError("unknown B subtype %r" % sub)
            n = struct.unpack_from("<I", buf, p + 1)[0]
            p += 5 + n * _B_SIZE[sub]
        else:
            raise BamError("unknown tag type %r" % ty)
    return tags


def _parse_record(buf):
    ref_id, pos, l_name, mapq, _bin, n_cig, flag, l_seq, _nr, _np, _tl = struct.unpack_from("<iiBBHHHiiii", buf, 0)
    p = 32
    r = Record()
    r.ref_id, r.reference_start, r.mapping_quality, r.flag, r.l_seq = ref_id, pos, mapq, flag, l_seq
    r.query_name = buf[p:p + l_name - 1].decode()
    p += l_name
    cig = np.frombuffer(buf, dtype="<u4", count=n_cig, offset=p)
    p += 4 * n_cig
    ops, lens = cig & 15, cig >> 4
    r.cigar = [(int(o), int(l)) for o, l in zip(ops, lens)]
    ref_span = int(sum(int(l) for o, l in zip(ops, lens) if _CIGAR_REF[o]))
    lead = trail = 0
    r.hard_clipped = bool(n_cig and (ops[0] == 5 or ops[-1] == 5))
    for o, l in zip(ops, lens):       # leading soft clip (hard clips are not in SEQ)
        if o == 4:
            lead += int(l)
        elif o != 5:
            break
    for o, l in zip(ops[::-1], lens[::-1]):
        if o == 4:
            trail += int(l)
        elif o != 5:
            break
    r.reference_end = pos + ref_span
    r.query_alignment_start = lead
    r.query_alignment_end = l_seq - trail
    nb = (l_seq + 1) // 2
    r.seq_nibbles = buf[p:p + nb]
    p += nb
    r.qual = buf[p:p + l_seq]
    p += l_seq
    r.tags = _parse_tags(buf, p, len(buf))
    return r


class BamReader:
    def __init__(self, path):
        self.path = path
        self.bg = _BgzfReader(path)
        self.bg.seek(0)
        if self.bg.read(4) != b"BAM\x01":
            raise BamError("%s is not a BAM file" % path)
        l_text = struct.unpack("<i", self.bg.read(4))[0]
        self.header_text = self.bg.read(l_text).rstrip(b"\0").decode()
        n_ref = struct.unpack("<i", self.bg.read(4))[0]
        self.references, self.lengths = [], []
        for _ in range(n_ref):
            l_name = struct.unpack("<i", self.bg.read(4))[0]
            self.references.append(self.bg.read(l_name)[:-1].decode())
            self.lengths.append(struct.unpack("<i", self.bg.read(4))[0])
        self.first_record = self.bg.tell()
        self.index_kind, self.index = "none", None
        for ip, kind in index_paths(path):
            if os.path.exists(ip):
                self.index_kind = kind
                self.index = _load_bai(ip, n_ref) if kind == "bai" else _load_csi(ip, self.references, self.lengths, path)
                break

    def close(self):
        self.bg.close()

    def _records_from(self, voffset):
        self.bg.seek(voffset)
        while True:
            head = self.bg.read(4)
            if len(head) < 4:
                return
            size = struct.unpack("<i", head)[0]
            yield _parse_record(self.bg.read(size))

    def seek_offset(self, rid, pos):
        """the virtual offset a fetch from pos of contig rid reads from; None: the index knows no record of the contig"""
        if self.index is None:
            return self.first_record
        if self.index_kind == "csi":
            return self.index.seek(rid, pos)
        lin = self.index[rid]
        if lin is None:
            return None
        w = min(pos >> 14, len(lin) - 1) if len(lin) else -1
        voff = None
        while w >= 0 and voff is None:   # windows nothing overlaps have offset 0
            voff = lin[w] or None
            w -= 1
        return self.first_record if voff is None else voff

    def fetch(self, chrom=None, start=None, end=None):
        """records overlapping [start, end) of chrom in file order (whole contig when start is None)"""
        if chrom is None:
            yield from self._records_from(self.first_record)
            return
        if chrom not in self.references:
            raise ValueError("invalid contig %r" % chrom)
        rid = self.references.index(chrom)
        lo = 0 if start is None else max(int(start), 0)
        hi = self.lengths[rid] if end is None else int(end)
        voff = self.seek_offset(rid, lo)
        if voff is None:
            return
        for r in self._records_from(voff):
            if r.ref_id != rid:
                if r.ref_id > rid or r.ref_id < 0:
                    return
                continue
            if r.reference_start >= hi:
                return
            rend = r.reference_end if r.reference_end > r.reference_start else r.reference_start + 1
            if rend > lo:
                yield r

    def count(self, chrom=None, start=None, end=None):
        return sum(1 for _ in self.fetch(chrom, start, end))


def _load_bai(path, n_ref):
    """-> per reference: list of linear-index virtual offsets (or None when the contig has no reads)"""
    try:
        data = open(path, "rb").read()
    except OSError:
        return None
    if data[:4] != b"BAI\x01":
        raise BamError("%s is not a BAI index" % path)
    p = 8
    out = []
    for _ in range(struct.unpack_from("<i", data, 4)[0]):
        n_bin = struct.unpack_from("<i", data, p)[0]
        p += 4
        for _b in range(n_bin):
            _bin, n_chunk = struct.unpack_from("<Ii", data, p)
            p += 8 + 16 * n_chunk
        n_intv = struct.unpack_from("<i", data, p)[0]
        p += 4
        lin = list(struct.unpack_from("<%dQ" % n_intv, data, p)) if n_intv else []
        p += 8 * n_intv
        out.append(lin if (n_bin or n_intv) else None)
    while len(out) < n_ref:
        out.append(None)
    return out


def index_paths(path):
    """[(index path, "bai" | "csi"), ...] in the order the readers look for them"""
    out = [(path + ".bai", "bai"), (path + ".csi", "csi")]
    if len(path) > 4 and path.endswith(".bam"):
        out += [(path[:-4] + ".bai", "bai"), (path[:-4] + ".csi", "csi")]
    return out


def _bin_first(level):
    return ((1 << (3 * level)) - 1) // 7


def _bin_level(b):
    lv = 0
    while b >= _bin_first(lv + 1):
        lv += 1
    return lv


def bin_start(b, min_shift=14, depth=5):
    """first reference position of bin b of the (min_shift, depth) binning scheme (SAM spec 5.3)"""
    lv = _bin_level(b)
    return (b - _bin_first(lv)) << (min_shift + 3 * (depth - lv))


def pseudo_bin(depth):
    return _bin_first(depth + 1) + 1


class CsiIndex:
    """a parsed CSI: min_shift, depth and per reference {bin: (loffset, [(beg, end), ...])} (None: no bins), the
    pseudo-bin and bins without chunks left out"""

    def __init__(self, min_shift, depth, refs):
        self.min_shift, self.depth, self.refs = min_shift, depth, refs

    def seek(self, rid, pos):
        """htslib's hts_itr_query: the loffset of the leaf bin that holds pos, else of its nearest left sibling, else of
        its parent, and so on up; without one, the contig's first chunk.  None: no record of the contig."""
        bins = self.refs[rid] if rid < len(self.refs) else None
        if not bins:
            return None
        top = (1 << (self.min_shift + 3 * self.depth)) - 1
        b = _bin_first(self.depth) + (min(pos, top) >> self.min_shift)
        while True:
            if b in bins and bins[b][0]:
                return bins[b][0]
            if b == 0:
                break
            first = (((b - 1) >> 3) << 3) + 1
            b = b - 1 if b > first else (b - 1) >> 3
        return min(c[0] for _l, ch in bins.values() for c in ch)


def _load_csi(path, names, lengths, bam_path):
    """-> CsiIndex; BamError naming the file for anything that cannot be read"""
    def bad(why):
        return BamError("%s: %s" % (path, why))
    raw = open(path, "rb").read()
    f, data = io.BytesIO(raw), []
    try:
        while True:
            at = f.tell()
            size, payload = _read_block(f)
            if size == 0:
                break
            if len(raw) < at + size or struct.unpack_from("<II", raw, at + size - 8) != (zlib.crc32(payload), len(payload)):
                raise BamError("bad block")
            data.append(payload)
    except (BamError, struct.error, zlib.error) as e:
        raise BamError("%s is not a BGZF-compressed CSI index (%s)" % (path, e))
    data = b"".join(data)
    bam_size = os.path.getsize(bam_path)
    if len(data) < 16 or data[:4] != b"CSI\x01":
        raise BamError("%s is not a CSI index" % path)
    min_shift, depth, l_aux = struct.unpack_from("<iii", data, 4)
    if min_shift < 1 or depth < 0 or depth > 10 or min_shift + 3 * depth > 62:
        raise bad("unsupported min_shift %d / depth %d" % (min_shift, depth))
    for name, ln in zip(names, lengths):
        if ln > 1 << (min_shift + 3 * depth):
            raise bad("min_shift %d and depth %d cover %d positions, %s has %d" % (min_shift, depth, 1 << (min_shift + 3 * depth), name, ln))
    p = 16 + l_aux
    if l_aux < 0 or p + 4 > len(data):
        raise bad("l_aux %d runs past the end of the index" % l_aux)
    pseudo = pseudo_bin(depth)

    def take(fmt, what):
        nonlocal p
        if p + struct.calcsize(fmt) > len(data):
            raise bad("truncated at byte %d (%s)" % (p, what))
        v = struct.unpack_from(fmt, data, p)
        p += struct.calcsize(fmt)
        return v

    n_ref, = take("<i", "n_ref")
    if n_ref < 0:
        raise bad("n_ref %d" % n_ref)
    refs = []
    for _ in range(n_ref):
        n_bin, = take("<i", "n_bin")
        if n_bin < 0 or n_bin * 16 > len(data) - p:
            raise bad("n_bin %d runs past the end of the index" % n_bin)
        bins = {}
        for _b in range(n_bin):
            b, loff, n_chunk = take("<IQi", "bin")
            if b > pseudo or b == pseudo - 1:  # pseudo - 1 is past the last level
                raise bad("bin %d past the pseudo-bin %d" % (b, pseudo))
            if b != pseudo and loff >> 16 >= bam_size:
                raise bad("loffset of bin %d points past the end of the BAM" % b)
            if n_chunk < 0 or n_chunk * 16 > len(data) - p:
                raise bad("n_chunk %d of bin %d runs past the end of the index" % (n_chunk, b))
            chunks = [struct.unpack_from("<QQ", data, p + 16 * c) for c in range(n_chunk)]
            p += 16 * n_chunk
            if b == pseudo:
                continue
            for c, (beg, end) in enumerate(chunks):
                if beg > end:
                    raise bad("chunk %d of bin %d begins after its end" % (c, b))
                if beg >> 16 >= bam_size:
                    raise bad("chunk %d of bin %d points past the end of the BAM" % (c, b))
            if chunks:
                loff0, ch0 = bins.get(b, (loff, []))
                bins[b] = (loff0, ch0 + chunks)
        refs.append(bins or None)
    while len(refs) < len(names):
        refs.append(None)
    return CsiIndex(min_shift, depth, refs)


# ------------------------------------------------------------------------------ region -> batch
def read_batch(reader, chrom, start, end, builder=None, refseq=None):
    """all records of `chrom` overlapping [start, end), packed (each record once, file order).

    Secondary records are dropped here: bamlib.BAM.__init__ skips them before anything else
    (src/himut/bamlib.py:17); supplementary records are kept, as the reference keeps them.
    A record's ops come from its cs:Z tag; a record without cs:Z but with MD:Z is decoded from CIGAR + MD
    (pack.parse_md: the same ops for the same alignment); a record with neither is decoded from CIGAR + refseq, the
    whole sequence of `chrom` (pack.parse_ref), when it is given, and rejected otherwise.
    """
    bb = builder or pack.BatchBuilder()
    for r in reader.fetch(chrom, start, end):
        if r.is_secondary:  # BAM.__init__ skips them everywhere (bamlib.py:17)
            continue
        if "cs" not in r.tags and "MD" not in r.tags and refseq is None:
            raise pack.BatchFormatError("%s has no cs:Z tag (the reference raises KeyError in BAM.__init__)" % r.query_name)
        # hard clips: pysam's query_sequence / query_alignment_start leave the clipped bases out (SEQ does not hold
        # them), so cs2tuple indexes consistently and the reference processes such records; so do we
        q = r.query_qualities
        if q is None:
            raise pack.BatchFormatError("%s has no base qualities" % r.query_name)
        bb.add(tstart=r.reference_start, tend=r.reference_end, qstart=r.query_alignment_start, qend=r.query_alignment_end,
               qseq=r.query_sequence, bq=bytes(q), mapq=r.mapping_quality, is_secondary=False, qname=r.query_name,
               cs=r.tags.get("cs"), cigar=r.cigar, md=r.tags.get("MD"), refseq=refseq)
    return bb.finish()


# ------------------------------------------------------------------------------ writer
def _reg2bin(beg, end, min_shift=14, depth=5):
    """the smallest bin of the (min_shift, depth) scheme that holds [beg, end) (htslib's hts_reg2bin)"""
    end -= 1
    sh = min_shift
    for lv in range(depth, 0, -1):
        if beg >> sh == end >> sh:
            return _bin_first(lv) + (beg >> sh)
        sh += 3
    return 0


def default_depth(lengths, min_shift=14):
    """htslib's choice of CSI depth: the smallest whose span holds the longest contig plus 256"""
    need, depth = max(lengths, default=0) + 256, 0
    while (1 << (min_shift + 3 * depth)) < need:
        depth += 1
    return depth


def _bgzf_block(chunk, level):
    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    comp = c.compress(chunk) + c.flush()
    return (b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", len(comp) + 25)
            + comp + struct.pack("<II", zlib.crc32(chunk), len(chunk)))


class BamWriter:
    """coordinate-sorted BAM + index writer; records must be added in sorted order.  index="bai" writes <path>.bai
    (refused for a contig longer than 2^29); index="csi" writes <path>.csi as htslib writes it, with min_shift and
    depth (None: default_depth)."""

    def __init__(self, path, references, header_extra="@RG\tID:rg\tSM:synth\n", level=1, index="bai", min_shift=14, depth=None):
        self.path, self.refs, self.level = path, list(references), level
        if index not in ("bai", "csi"):
            raise ValueError("index must be 'bai' or 'csi'")
        if index == "bai" and any(ln > BAI_MAX_LEN for _n, ln in self.refs):
            raise ValueError("a BAI cannot index a contig longer than 2^29: use index='csi'")
        self.index = index
        self.min_shift = min_shift if index == "csi" else 14
        self.depth = 5 if index == "bai" else (default_depth([ln for _n, ln in self.refs], min_shift) if depth is None else depth)
        if (1 << (self.min_shift + 3 * self.depth)) < max([ln for _n, ln in self.refs], default=0):
            raise ValueError("min_shift %d and depth %d do not cover the longest contig" % (self.min_shift, self.depth))
        self.f = open(path, "wb")
        self.coff = 0
        self.buf = bytearray()
        text = "@HD\tVN:1.6\tSO:coordinate\n" + "".join("@SQ\tSN:%s\tLN:%d\n" % r for r in self.refs) + header_extra
        head = bytearray(b"BAM\x01") + struct.pack("<i", len(text)) + text.encode() + struct.pack("<i", len(self.refs))
        for name, ln in self.refs:
            head += struct.pack("<i", len(name) + 1) + name.encode() + b"\0" + struct.pack("<i", ln)
        self._write(bytes(head))
        self._flush()
        self.bins = [dict() for _ in self.refs]
        self.lin = [[] for _ in self.refs]
        self.n_mapped = [0] * len(self.refs)

    def _emit_block(self, chunk):
        block = _bgzf_block(chunk, self.level)
        self.f.write(block)
        self.coff += len(block)

    def _flush(self, everything=True):
        """cut the pending bytes into <= 0xFF00-byte blocks; the tail stays pending unless `everything`"""
        while len(self.buf) >= 0xFF00 or (everything and self.buf):
            chunk = bytes(self.buf[:0xFF00])
            del self.buf[:0xFF00]
            self._emit_block(chunk)

    def _write(self, b):
        self.buf += b

    def add(self, ref_id, pos, qname, flag, mapq, cigar, seq, qual, tags):
        """cigar: list of (op, len); seq: ASCII str; qual: bytes; tags: list of (tag, type, value), type one of
        A Z H c C s S i I f, or B with value (subtype, list of numbers)"""
        v0 = (self.coff << 16) | len(self.buf)
        ref_span = sum(l for o, l in cigar if _CIGAR_REF[o])
        end = pos + max(ref_span, 1)
        l_seq = len(seq)
        codes = np.array([_SEQ_DEC.index(c) if c in _SEQ_DEC else 15 for c in seq.upper()], np.uint8)
        if l_seq % 2:
            codes = np.concatenate([codes, np.zeros(1, np.uint8)])
        packed = ((codes[0::2] << 4) | codes[1::2]).astype(np.uint8).tobytes()
        bai_bin = _reg2bin(pos, end) if end - 1 < BAI_MAX_LEN else 4680  # no decoder here reads it: past 2^29 it cannot be right
        body = struct.pack("<iiBBHHHiiii", ref_id, pos, len(qname) + 1, mapq, bai_bin, len(cigar), flag, l_seq, -1, -1, 0)
        body += qname.encode() + b"\0" + b"".join(struct.pack("<I", (l << 4) | o) for o, l in cigar) + packed + bytes(qual)
        for tag, ty, val in tags:
            body += tag.encode() + ty.encode()
            if ty in ("Z", "H"):
                body += val.encode() + b"\0"
            elif ty == "A":
                body += val.encode()
            elif ty == "B":
                sub, vals = val
                body += sub.encode() + struct.pack("<I%d%s" % (len(vals), _TAG_FMT[sub]), len(vals), *vals)
            elif ty in _TAG_FMT:
                body += struct.pack("<" + _TAG_FMT[ty], val)
            else:
                raise ValueError("unknown tag type %r" % ty)
        rec = struct.pack("<i", len(body)) + body
        self.buf += rec
        self._flush(everything=False)  # pending tail < 0xFF00, so offsets stay exact
        v1 = (self.coff << 16) | len(self.buf)
        if ref_id >= 0:
            self.bins[ref_id].setdefault(_reg2bin(pos, end, self.min_shift, self.depth), []).append((v0, v1))
            self.n_mapped[ref_id] += 1
            lin = self.lin[ref_id]
            for w in range(pos >> self.min_shift, ((end - 1) >> self.min_shift) + 1):
                while len(lin) <= w:
                    lin.append(0)
                if lin[w] == 0:
                    lin[w] = v0

    def close(self):
        self._flush()
        self.f.write(_BGZF_EOF)
        self.f.close()
        if self.index == "csi":
            self._write_csi()
            return
        with open(self.path + ".bai", "wb") as f:
            f.write(b"BAI\x01" + struct.pack("<i", len(self.refs)))
            for bins, lin in zip(self.bins, self.lin):
                f.write(struct.pack("<i", len(bins)))
                for b, chunks in sorted(bins.items()):
                    f.write(struct.pack("<Ii", b, len(chunks)))
                    for beg, end in chunks:
                        f.write(struct.pack("<QQ", beg, end))
                # fill empty linear windows with the next known offset (htslib does the same backwards)
                f.write(struct.pack("<i", len(lin)))
                last = 0
                filled = []
                for v in lin:
                    if v:
                        last = v
                    filled.append(v or last)
                f.write(struct.pack("<%dQ" % len(filled), *filled))
            f.write(struct.pack("<Q", 0))

    def _write_csi(self):
        ms, depth = self.min_shift, self.depth
        out = bytearray(b"CSI\x01" + struct.pack("<iiii", ms, depth, 0, len(self.refs)))
        for bins, lin, n_mapped in zip(self.bins, self.lin, self.n_mapped):
            # htslib's linear index (update_loff): windows before the first entry take the contig's first record, later
            # empty ones the entry to their left; a bin's loffset is the entry of its first window
            first = min((ch[0][0] for ch in bins.values()), default=0)
            filled, last = [], first
            for v in lin:
                last = v or last
                filled.append(last)
            out += struct.pack("<i", len(bins) + (1 if bins else 0))
            for b, chunks in sorted(bins.items()):
                merged = []  # adjacent records of one bin share a chunk, as htslib writes them
                for beg, end in chunks:
                    if merged and merged[-1][1] == beg:
                        merged[-1] = (merged[-1][0], end)
                    else:
                        merged.append((beg, end))
                bot = bin_start(b, ms, depth) >> ms
                out += struct.pack("<IQi", b, filled[bot] if bot < len(filled) else 0, len(merged))
                out += b"".join(struct.pack("<QQ", *c) for c in merged)
            if bins:  # the pseudo-bin: first and last offsets of the contig, mapped and unmapped record counts
                last_end = max(ch[-1][1] for ch in bins.values())
                out += struct.pack("<IQi", pseudo_bin(depth), 0, 2) + struct.pack("<QQQQ", first, last_end, n_mapped, 0)
        out += struct.pack("<Q", 0)  # n_no_coor
        with open(self.path + ".csi", "wb") as f:
            for k in range(0, len(out), 0xFF00):
                f.write(_bgzf_block(bytes(out[k:k + 0xFF00]), self.level))
            f.write(_BGZF_EOF)


TAGS = ("cs", "md", "md_eqx", "eqx", "m")


def write_batch_bam(path, chrom, contig_len, batch, sample="synth", tags="cs", **index):
    """ReadBatch -> coordinate-sorted BAM + BAI, tp:A:P, for tests and tools.  tags: "cs" writes cs:Z short form
    with a =/X CIGAR; "md" writes MD:Z and no cs with an M CIGAR; "md_eqx" MD:Z with the =/X CIGAR; "eqx" the =/X
    CIGAR and neither tag; "m" the M CIGAR and neither tag (these two decode with the contig's reference sequence)"""
    write_batches_bam(path, [(chrom, contig_len, batch)], sample, tags, **index)


def write_batches_bam(path, contigs, sample="synth", tags="cs", **index):
    """[(chrom, contig_len, ReadBatch), ...] -> one coordinate-sorted BAM + BAI (index, min_shift, depth: BamWriter's)"""
    w = BamWriter(path, [(c, n) for c, n, _ in contigs], header_extra="@RG\tID:rg\tSM:%s\n" % sample, **index)
    for rid, (_c, _n, batch) in enumerate(contigs):
        _add_batch(w, rid, batch, tags)
    w.close()


def _add_batch(w, rid, batch, tags="cs"):
    if tags not in TAGS:
        raise ValueError("tags must be one of %s" % (TAGS,))
    m_op, x_op = (0, 0) if tags in ("md", "m") else (7, 8)
    aln_tag = {"cs": "cs", "md": "MD", "md_eqx": "MD"}.get(tags)
    for r in range(batch.n_reads):
        ql = int(batch.qlen[r])
        so, bo, oo = int(batch.seq_off[r]), int(batch.bq_off[r]), int(batch.op_off[r])
        packed = batch.seq[so:so + (ql + 3) // 4]
        codes = ((packed[:, None] >> np.array([0, 2, 4, 6], np.uint8)) & 3).reshape(-1)[:ql]
        qseq = "".join("ATGC"[c] for c in codes)
        ops = batch.ops[oo:oo + int(batch.n_ops[r])]
        qstart = int(batch.qstart[r])
        cs, cigar, q = [], [], qstart
        md, md_run = [], 0  # MD: the matched bases since the last event, then the event (deleted bases as N)
        if qstart:
            cigar.append((4, qstart))
        for wd in ops:
            kind, val = int(wd) & 3, int(wd) >> 2
            if kind == abi.OP_MATCH:
                cs.append(":%d" % val); cigar.append((m_op, val)); q += val
                md_run += val
            elif kind == abi.OP_SUB:
                cs.append("*%s%s" % ("atgcn"[val & 7], "atgcn"[(val >> 3) & 7])); cigar.append((x_op, 1)); q += 1
                md.append("%d%s" % (md_run, "ATGCN"[val & 7])); md_run = 0
            elif kind == abi.OP_INS:
                cs.append("+" + qseq[q:q + val].lower()); cigar.append((1, val)); q += val
            else:
                cs.append("-" + "n" * val); cigar.append((2, val))
                md.append("%d^%s" % (md_run, "N" * val)); md_run = 0
        if ql - q:
            cigar.append((4, ql - q))
        merged = []
        for o, l in cigar:
            if merged and merged[-1][0] == o:
                merged[-1] = (o, merged[-1][1] + l)
            else:
                merged.append((o, l))
        flag = 0x100 if (batch.flags[r] & abi.READ_SECONDARY) else 0
        w.add(rid, int(batch.tstart[r]), "read%d" % int(batch.qname_id[r]), flag, int(batch.mapq[r]), merged, qseq,
              batch.bq[bo:bo + ql].tobytes(),
              ([("cs", "Z", "".join(cs)) if aln_tag == "cs" else ("MD", "Z", "".join(md) + "%d" % md_run)] if aln_tag else [])
              + [("tp", "A", "P")])
