"""Minimal BAM / BGZF / BAI reader and writer (pure Python + zlib).

pysam / htslib are not available in this image (SURVEY.md §0.4), and the worker mirrors need the
records of a region as a packed ReadBatch rather than as Python objects anyway.  The reader
implements what the reference touches through pysam (SURVEY.md §8b): header text, @SQ table,
fetch(chrom, start, end) — records overlapping the 0-based half-open window, in file order,
secondary / supplementary included — and the per-record fields reference_start/end,
query_alignment_start/end, query_sequence, query_qualities, mapping_quality, flag, cs:Z, tp:A, and
beyond it the CIGAR and MD:Z (records without cs:Z are decoded from CIGAR + MD, pack.parse_md).
The writer exists for tests and for the synthetic-data tools (coordinate-sorted BAM + .bai).
"""
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
            n = struct.unpack_from("<I", buf, p + 1)[0]
            p += 5 + n * {"c": 1, "C": 1, "s": 2, "S": 2, "i": 4, "I": 4, "f": 4}[sub]
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
        self.index = _load_bai(path + ".bai", n_ref)

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
        voff = self.first_record
        if self.index is not None:
            lin = self.index[rid]
            if lin is None:
                return
            w = min(lo >> 14, len(lin) - 1) if len(lin) else -1
            voff = None
            while w >= 0 and voff is None:   # windows nothing overlaps have offset 0
                voff = lin[w] or None
                w -= 1
            if voff is None:
                voff = self.first_record
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


# ------------------------------------------------------------------------------ region -> batch
def read_batch(reader, chrom, start, end, builder=None):
    """all records of `chrom` overlapping [start, end), packed (each record once, file order).

    Secondary records are dropped here: bamlib.BAM.__init__ skips them before anything else
    (src/himut/bamlib.py:17); supplementary records are kept, as the reference keeps them.
    A record's ops come from its cs:Z tag; a record without cs:Z but with MD:Z is decoded from CIGAR + MD
    (pack.parse_md: the same ops for the same alignment); a record with neither is rejected.
    """
    bb = builder or pack.BatchBuilder()
    for r in reader.fetch(chrom, start, end):
        if r.is_secondary:  # BAM.__init__ skips them everywhere (bamlib.py:17)
            continue
        if "cs" not in r.tags and "MD" not in r.tags:
            raise pack.BatchFormatError("%s has no cs:Z tag (the reference raises KeyError in BAM.__init__)" % r.query_name)
        # hard clips: pysam's query_sequence / query_alignment_start leave the clipped bases out (SEQ does not hold
        # them), so cs2tuple indexes consistently and the reference processes such records; so do we
        q = r.query_qualities
        if q is None:
            raise pack.BatchFormatError("%s has no base qualities" % r.query_name)
        bb.add(tstart=r.reference_start, tend=r.reference_end, qstart=r.query_alignment_start, qend=r.query_alignment_end,
               qseq=r.query_sequence, bq=bytes(q), mapq=r.mapping_quality, is_secondary=False, qname=r.query_name,
               cs=r.tags.get("cs"), cigar=r.cigar, md=r.tags.get("MD"))
    return bb.finish()


# ------------------------------------------------------------------------------ writer
def _reg2bin(beg, end):
    end -= 1
    if beg >> 14 == end >> 14:
        return ((1 << 15) - 1) // 7 + (beg >> 14)
    if beg >> 17 == end >> 17:
        return ((1 << 12) - 1) // 7 + (beg >> 17)
    if beg >> 20 == end >> 20:
        return ((1 << 9) - 1) // 7 + (beg >> 20)
    if beg >> 23 == end >> 23:
        return ((1 << 6) - 1) // 7 + (beg >> 23)
    if beg >> 26 == end >> 26:
        return ((1 << 3) - 1) // 7 + (beg >> 26)
    return 0


class BamWriter:
    """coordinate-sorted BAM + BAI writer; records must be added in sorted order"""

    def __init__(self, path, references, header_extra="@RG\tID:rg\tSM:synth\n", level=1):
        self.path, self.refs, self.level = path, list(references), level
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

    def _emit_block(self, chunk):
        c = zlib.compressobj(self.level, zlib.DEFLATED, -15)
        comp = c.compress(chunk) + c.flush()
        block = (b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", len(comp) + 25)
                 + comp + struct.pack("<II", zlib.crc32(chunk), len(chunk)))
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
        """cigar: list of (op, len); seq: ASCII str; qual: bytes; tags: list of (tag, type, value)"""
        v0 = (self.coff << 16) | len(self.buf)
        ref_span = sum(l for o, l in cigar if _CIGAR_REF[o])
        end = pos + max(ref_span, 1)
        l_seq = len(seq)
        codes = np.array([_SEQ_DEC.index(c) if c in _SEQ_DEC else 15 for c in seq.upper()], np.uint8)
        if l_seq % 2:
            codes = np.concatenate([codes, np.zeros(1, np.uint8)])
        packed = ((codes[0::2] << 4) | codes[1::2]).astype(np.uint8).tobytes()
        body = struct.pack("<iiBBHHHiiii", ref_id, pos, len(qname) + 1, mapq, _reg2bin(pos, end), len(cigar), flag, l_seq, -1, -1, 0)
        body += qname.encode() + b"\0" + b"".join(struct.pack("<I", (l << 4) | o) for o, l in cigar) + packed + bytes(qual)
        for tag, ty, val in tags:
            if ty == "Z":
                body += tag.encode() + b"Z" + val.encode() + b"\0"
            elif ty == "A":
                body += tag.encode() + b"A" + val.encode()
            elif ty == "i":
                body += tag.encode() + b"i" + struct.pack("<i", val)
        rec = struct.pack("<i", len(body)) + body
        self.buf += rec
        self._flush(everything=False)  # pending tail < 0xFF00, so offsets stay exact
        v1 = (self.coff << 16) | len(self.buf)
        if ref_id >= 0:
            self.bins[ref_id].setdefault(_reg2bin(pos, end), []).append((v0, v1))
            lin = self.lin[ref_id]
            for w in range(pos >> 14, ((end - 1) >> 14) + 1):
                while len(lin) <= w:
                    lin.append(0)
                if lin[w] == 0:
                    lin[w] = v0

    def close(self):
        self._flush()
        self.f.write(_BGZF_EOF)
        self.f.close()
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


TAGS = ("cs", "md", "md_eqx")


def write_batch_bam(path, chrom, contig_len, batch, sample="synth", tags="cs"):
    """ReadBatch -> coordinate-sorted BAM + BAI, tp:A:P, for tests and tools.  tags: "cs" writes cs:Z short form
    with a =/X CIGAR; "md" writes MD:Z and no cs with an M CIGAR; "md_eqx" MD:Z with the =/X CIGAR"""
    write_batches_bam(path, [(chrom, contig_len, batch)], sample, tags)


def write_batches_bam(path, contigs, sample="synth", tags="cs"):
    """[(chrom, contig_len, ReadBatch), ...] -> one coordinate-sorted BAM + BAI"""
    w = BamWriter(path, [(c, n) for c, n, _ in contigs], header_extra="@RG\tID:rg\tSM:%s\n" % sample)
    for rid, (_c, _n, batch) in enumerate(contigs):
        _add_batch(w, rid, batch, tags)
    w.close()


def _add_batch(w, rid, batch, tags="cs"):
    if tags not in TAGS:
        raise ValueError("tags must be one of %s" % (TAGS,))
    m_op, x_op = (0, 0) if tags == "md" else (7, 8)
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
              [("cs", "Z", "".join(cs)) if tags == "cs" else ("MD", "Z", "".join(md) + "%d" % md_run), ("tp", "A", "P")])
