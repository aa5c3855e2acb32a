"""One contig of an uncompressed FASTA file, for the decoders' CIGAR + reference path (pack.parse_ref).

Records with neither cs:Z nor MD:Z carry only where the read aligns; the reference base at each aligned position comes
from the FASTA the reads were aligned to.  The contig is read through <fasta>.fai when that index exists (one seek and
one read), by scanning the file for its header otherwise.  The contig name is the first word of the header line, as
samtools faidx and pyfastx take it.  Case is kept: the decoders compare bases case-insensitively.
"""
import mmap
import os


def _check_plain(path):
    with open(path, "rb") as f:
        if f.read(2) == b"\x1f\x8b":
            raise ValueError("%s is gzip / bgzip compressed: decompress it (e.g. `gzip -dc %s > ref.fa`) and pass the "
                             "plain FASTA" % (path, os.path.basename(path)))


def _from_fai(path, fai, name):
    with open(fai) as f:
        for line in f:
            cols = line.rstrip("\n").split("\t")
            if cols[0] != name:
                continue
            length, offset, line_bases, line_width = (int(c) for c in cols[1:5])
            if length == 0:
                return b""
            n_lines = (length + line_bases - 1) // line_bases
            with open(path, "rb") as fa:
                fa.seek(offset)
                raw = fa.read(n_lines * line_width)  # may reach into the next record: only `length` bases are kept
            seq = raw.replace(b"\n", b"").replace(b"\r", b"")[:length]
            if len(seq) != length:
                raise ValueError("%s ends inside contig %s: its .fai promises %d bases, the file holds %d"
                                 % (path, name, length, len(seq)))
            return seq
    return None


def _scan(path, name):
    with open(path, "rb") as f:
        if os.fstat(f.fileno()).st_size == 0:
            return None
        with mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ) as mm:
            head = 0 if mm[:1] == b">" else mm.find(b"\n>")
            if head < 0:
                return None
            head += head > 0  # the ">" after the newline
            want = name.encode()
            while True:
                eol = mm.find(b"\n", head)
                eol = len(mm) if eol < 0 else eol
                words = mm[head + 1:eol].split()
                nxt = mm.find(b"\n>", eol)
                end = len(mm) if nxt < 0 else nxt
                if words and words[0] == want:
                    return mm[eol + 1:end].replace(b"\n", b"").replace(b"\r", b"")
                if nxt < 0:
                    return None
                head = nxt + 1


def write_fasta(path, contigs, width=60):
    """[(name, sequence bytes or str), ...] -> a FASTA with lines of `width` bases (tools: the synthetic contigs)"""
    with open(path, "w") as f:
        for name, seq in contigs:
            seq = seq.decode() if isinstance(seq, (bytes, bytearray)) else seq
            f.write(">%s\n" % name + "".join(seq[i:i + width] + "\n" for i in range(0, len(seq), width)))


def load_contig(path, name, length=None):
    """the sequence of contig `name` in the FASTA at `path`, as bytes.  length: the contig's length in the BAM header
    (@SQ LN); a sequence of another length is an error, so that a FASTA of another reference build fails here instead
    of turning every base into a SUB."""
    _check_plain(path)
    fai = path + ".fai"
    seq = _from_fai(path, fai, name) if os.path.exists(fai) else _scan(path, name)
    if seq is None:
        raise ValueError("contig %s is not in the FASTA %s" % (name, path))
    if length is not None and len(seq) != int(length):
        raise ValueError("contig %s has %d bases in the FASTA %s but %d in the BAM header (@SQ LN): is it the reference "
                         "the reads were aligned to?" % (name, len(seq), path, int(length)))
    return seq
