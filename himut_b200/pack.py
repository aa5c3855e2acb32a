"""Decoded alignment records -> packed ReadBatch (the host half of the expansion step).

parse_cs turns a minimap2 cs:Z tag into the u32 op stream of include/himut_b200.h with the
token grammar of the reference's cslib.cs2lst / cs2tuple (src/himut/cslib.py:7-44): ":n" and
"=SEQ" matches, "*xy" substitutions, "+seq" insertions, "-seq" deletions, case-insensitive.
Inputs the reference would crash on are rejected here, loudly, instead of reaching a kernel:
read bases outside ACGT under a match / substitution (KeyError at caller.py:57,62), "~"
introns, a cs tag whose spans disagree with the CIGAR-derived coordinates.

parse_md gives the same ops from a CIGAR plus an MD:Z tag, for records without cs:Z (pbmm2 output,
minimap2 without --cs; `samtools calmd` adds MD to any BAM).  The reference reads cs only and
raises KeyError on such records; for the same alignment both tags give the same op stream.

parse_ref gives the same ops from the CIGAR and the contig's reference sequence, for records with
neither tag (what minimap2 writes without --cs or --MD, and what pbmm2 writes).
"""
import re

import numpy as np

from . import abi

_CS_TOKEN = re.compile(r"(:[0-9]+|\*[a-zA-Z][a-zA-Z]|[=\+\-][A-Za-z]+)")
_CODE = np.full(256, 255, np.uint8)
for _b, _c in abi.BASE2CODE.items():
    _CODE[ord(_b)] = _c
    _CODE[ord(_b.lower())] = _c


class BatchFormatError(ValueError):
    pass


# CIGAR + MD:Z.  The messages are those of csrc/bamerr.h, which both native decoders use, so that the three
# implementations reject a record with the same words.
_MD_GRAMMAR = re.compile(r"[0-9]+(?:(?:[A-Za-z]|\^[A-Za-z]+)[0-9]+)*")
_MD_PART = re.compile(r"[0-9]+|\^[A-Za-z]+|[A-Za-z]")
MD_ERR = {
    "md_token": "%s: unsupported MD:Z token (%d)",
    "md_span": "%s: MD:Z and CIGAR disagree at reference offset %d",
    "cigar_op": "%s: unsupported CIGAR op (N, P, or a clip inside the alignment) at CIGAR index %d",
    "span_qry": "%s: cs query span != aligned query span (%d)",
    "n_match": "%s: read base outside A/C/G/T under a cs match (reference: KeyError) (%d)",
    "sub_n": "%s: substitution to a base outside A/C/G/T (the reference pileup raises KeyError) (%d)",
}
_M, _I, _D, _S, _H, _EQ, _X = 0, 1, 2, 4, 5, 7, 8
# CIGAR + reference: the messages of the two checks only this path makes (csrc/bamerr.h); the others are MD_ERR's
REF_ERR = {
    "ref_end": "%s: alignment runs past the end of the reference sequence (%d)",
    "ref_span": "%s: CIGAR and the reference sequence disagree at reference offset %d",
}
# reference bytes -> codes, case-insensitive; anything outside A/C/G/T (N, IUPAC codes) is BASE_N, as minimap2 writes it
_REF_CODE = np.full(256, abi.BASE_N, np.uint8)
for _b, _c in abi.BASE2CODE.items():
    _REF_CODE[ord(_b)] = _c
    _REF_CODE[ord(_b.lower())] = _c


def _fail(key, qname, arg):
    raise BatchFormatError((MD_ERR.get(key) or REF_ERR[key]) % (qname, arg))


def _check_cigar(cigar, qseq, qname):
    """the CIGAR checks parse_md and parse_ref share: N, P, codes past X and S / H between the first and the last
    aligned op are unsupported; the CIGAR's query length must be len(qseq)"""
    core = [i for i, (o, _l) in enumerate(cigar) if o not in (_S, _H)]
    qcore = qclip = 0
    for i, (o, l) in enumerate(cigar):
        if o in (_S, _H):
            if core and core[0] < i < core[-1]:
                _fail("cigar_op", qname, i)
            qclip += l if o == _S else 0
        elif o in (_M, _I, _EQ, _X):
            qcore += l
        elif o != _D:
            _fail("cigar_op", qname, i)
    if qcore + qclip != len(qseq):
        _fail("span_qry", qname, qcore)


def parse_ref(cigar, refseq, tstart, qseq, qstart, qname="read"):
    """CIGAR [(op, len), ...] (BAM op codes) + the contig's reference sequence -> (ops, ref_span, query_span), the ops
    cs gives for the same alignment when the BAM agrees with its reference: one MATCH per maximal run of matched bases,
    SUB(reference base, read base) per mismatch, INS / DEL with the CIGAR length.  refseq: the whole contig (bytes or
    str), tstart the record's 0-based position; qseq the full read (soft clips included), qstart its leading soft clip.

    Checked in this order, each failure the first one the walk meets:
      - the CIGAR checks of parse_md (cigar_op, span_qry);
      - the alignment must lie inside the reference: tstart + reference span <= len(refseq) (ref_end), before any
        reference byte is read;
      - the walk.  Reference bases are case-insensitive, anything outside A/C/G/T is N.  M: a read base equal to an
        A/C/G/T reference base is matched, every other base is a SUB(reference base or N, read base), and a read base
        outside A/C/G/T there is rejected (sub_n, as cs "*xn").  =: the read base must be A/C/G/T (n_match) and equal
        to an A/C/G/T reference base (ref_span).  X: a read base outside A/C/G/T is rejected (sub_n), one equal to an
        A/C/G/T reference base disagrees with the CIGAR (ref_span); every other base is a SUB.
    A match run goes on across M / = / X and ends at a SUB, an I or a D; ops of length 0 are skipped.  Deleted
    reference bases are not read."""
    _check_cigar(cigar, qseq, qname)
    rspan = sum(l for o, l in cigar if o in (_M, _D, _EQ, _X))
    if tstart < 0 or tstart + rspan > len(refseq):
        _fail("ref_end", qname, tstart + rspan)
    rb = refseq.encode() if isinstance(refseq, str) else refseq
    rcodes = _REF_CODE[np.frombuffer(rb, dtype=np.uint8, count=rspan, offset=tstart)] if rspan else np.zeros(0, np.uint8)
    codes = _CODE[np.frombuffer(qseq.encode(), dtype=np.uint8)]
    ops, run, q, r = [], 0, qstart, 0

    def flush():
        nonlocal run
        if run:
            ops.append(abi.make_op(abi.OP_MATCH, run))
            run = 0

    for o, l in cigar:
        if l == 0 or o in (_S, _H):
            continue
        if o in (_M, _EQ, _X):
            rc, ac = rcodes[r:r + l], codes[q:q + l]
            match, bad = rc == ac, ac == 255  # rc is never 255: equal codes are A/C/G/T on both sides
            if o == _M:
                if bad.any():
                    _fail("sub_n", qname, q + int(np.argmax(bad)))
                subs = np.flatnonzero(~match)
            else:
                stop = (~match) if o == _EQ else (match | bad)
                if stop.any():
                    j = int(np.argmax(stop))
                    _fail(("n_match" if o == _EQ else "sub_n") if bad[j] else "ref_span", qname, (q + j) if bad[j] else (r + j))
                subs = np.arange(l) if o == _X else np.zeros(0, np.int64)
            last = -1
            for j in subs.tolist():
                run += j - last - 1
                flush()
                ops.append(abi.make_sub(int(rc[j]), int(ac[j])))
                last = j
            run += l - last - 1
            q += l; r += l
        elif o == _I:
            flush()
            ops.append(abi.make_op(abi.OP_INS, l))
            q += l
        else:
            flush()
            ops.append(abi.make_op(abi.OP_DEL, l))
            r += l
    flush()
    return ops, r, q - qstart


def parse_md(cigar, md, qseq, qstart, qname="read"):
    """CIGAR [(op, len), ...] (BAM op codes) + MD:Z -> (ops, ref_span, query_span), the ops cs gives for the
    same alignment: one MATCH per maximal run of matched bases, SUB(MD letter, read base) per mismatch, INS / DEL
    with the CIGAR length.  qseq is the full read (soft clips included), qstart its leading soft clip.

    Checked in this order, each failure the first one the walk meets:
      - CIGAR ops: N, P, codes past X, and S / H between the first and the last aligned op are unsupported
        (cs writes introns as "~", which parse_cs rejects too);
      - the CIGAR's query length must be len(qseq);
      - MD grammar [0-9]+(([A-Za-z]|^[A-Za-z]+)[0-9]+)*;
      - the walk: M, = and X take reference positions from MD; a match run goes on across M / = / X and across
        MD numbers and ends at a mismatch, an I or a D.  An MD letter is a SUB whose ref base is the letter (not
        A/C/G/T: N, as cs "*nx") and whose alt base is SEQ there (not A/C/G/T: rejected, as cs "*xn"); nothing
        checks that they differ, as for cs "*xy".  Matched read bases must be A/C/G/T.  "=" over an MD letter,
        "X" over an MD match, D without "^" and as many letters (any letters: only the length is kept), MD
        running out, or MD left at the end (a trailing 0 is fine) mean MD and CIGAR disagree.
    Ops of length 0 are skipped."""
    def fail(key, arg):
        _fail(key, qname, arg)

    _check_cigar(cigar, qseq, qname)
    m = _MD_GRAMMAR.match(md)
    if m is None or m.end() != len(md):
        fail("md_token", m.end() if m else 0)
    parts = _MD_PART.findall(md)
    mnum, ti = int(parts[0]), 1
    codes = _CODE[np.frombuffer(qseq.encode(), dtype=np.uint8)]
    ops, run, q, r = [], 0, qstart, 0

    def flush():
        nonlocal run
        if run:
            ops.append(abi.make_op(abi.OP_MATCH, run))
            run = 0

    for o, l in cigar:
        if l == 0 or o in (_S, _H):
            continue
        if o in (_M, _EQ, _X):
            k = 0
            while k < l:
                if mnum:
                    if o == _X:
                        fail("md_span", r)
                    t = min(mnum, l - k)
                    bad = np.flatnonzero(codes[q:q + t] == 255)
                    if bad.size:
                        fail("n_match", q + int(bad[0]))
                    run += t; mnum -= t; q += t; r += t; k += t
                else:
                    if ti >= len(parts) or parts[ti][0] == "^" or o == _EQ:
                        fail("md_span", r)
                    ref = abi.BASE2CODE.get(parts[ti].upper(), abi.BASE_N)
                    mnum, ti = int(parts[ti + 1]), ti + 2
                    if codes[q] == 255:
                        fail("sub_n", q)
                    flush()
                    ops.append(abi.make_sub(ref, int(codes[q])))
                    q += 1; r += 1; k += 1
        elif o == _I:
            flush()
            ops.append(abi.make_op(abi.OP_INS, l))
            q += l
        else:
            if mnum or ti >= len(parts) or parts[ti][0] != "^" or len(parts[ti]) - 1 != l:
                fail("md_span", r)
            mnum, ti = int(parts[ti + 1]), ti + 2
            flush()
            ops.append(abi.make_op(abi.OP_DEL, l))
            r += l
    flush()
    if mnum or ti < len(parts):
        fail("md_span", r)
    return ops, r, q - qstart


def parse_cs(cs, qseq, qstart):
    """-> (ops list[int], ref_span, query_span).  qseq is the full read (soft clips included)."""
    ops, rspan, q = [], 0, qstart
    pos = 0
    for m in _CS_TOKEN.finditer(cs):
        if m.start() != pos:
            raise BatchFormatError("unsupported cs token at %d in %r" % (pos, cs[pos:pos + 16]))
        pos = m.end()
        tok = m.group(0)
        head, body = tok[0], tok[1:]
        if head == ":":
            n = int(body)
            if n:
                ops.append(abi.make_op(abi.OP_MATCH, n))
            rspan += n; q += n
        elif head == "=":
            n = len(body)
            if qseq[q:q + n].upper() != body.upper():
                raise BatchFormatError("cs long-form bases disagree with SEQ at query %d" % q)
            ops.append(abi.make_op(abi.OP_MATCH, n))
            rspan += n; q += n
        elif head == "*":
            r, a = body[0].upper(), body[1].upper()
            if a not in abi.BASE2CODE:
                raise BatchFormatError("substitution to %r: the reference pileup needs A/C/G/T" % a)
            ops.append(abi.make_sub(abi.BASE2CODE.get(r, abi.BASE_N), abi.BASE2CODE[a]))
            rspan += 1; q += 1
        elif head == "+":
            ops.append(abi.make_op(abi.OP_INS, len(body)))
            q += len(body)
        else:
            ops.append(abi.make_op(abi.OP_DEL, len(body)))
            rspan += len(body)
    if pos != len(cs):
        raise BatchFormatError("unsupported cs token at %d in %r" % (pos, cs[pos:pos + 16]))
    # adjacent match tokens are kept apart: normcounts evaluates its mismatch window once per
    # match block (normcounts.py:82-87), so merging them would change edge cases
    return ops, rspan, q - qstart


def pack_seq(qseq_bytes, ops, qstart):
    """ASCII read -> 2-bit codes (4 per byte); bases under match ops must be ACGT"""
    codes = _CODE[np.frombuffer(qseq_bytes, dtype=np.uint8)]
    q = qstart
    for w in ops:
        kind, val = w & 3, w >> 2
        if kind == abi.OP_MATCH:
            if (codes[q:q + val] == 255).any():
                raise BatchFormatError("read base outside A/C/G/T under a cs match (reference: KeyError)")
            q += val
        elif kind == abi.OP_SUB:
            q += 1
        elif kind == abi.OP_INS:
            q += val
    codes = np.where(codes == 255, 0, codes).astype(np.uint8)
    pad = (-codes.size) % 4
    if pad:
        codes = np.concatenate([codes, np.zeros(pad, np.uint8)])
    c4 = codes.reshape(-1, 4)
    return (c4[:, 0] | (c4[:, 1] << 2) | (c4[:, 2] << 4) | (c4[:, 3] << 6)).astype(np.uint8)


class BatchBuilder:
    """accumulates decoded records of one contig, in file order"""

    def __init__(self):
        self.cols = {k: [] for k in ("tstart", "tend", "qstart", "qlen", "mapq", "flags", "qname_id",
                                     "seq_off", "bq_off", "op_off", "n_ops")}
        self.seq, self.bq, self.ops = [], [], []
        self.seq_n = self.bq_n = self.ops_n = 0
        self.qnames = {}

    def add(self, *, tstart, tend, qstart, qend, qseq, bq, mapq, is_secondary, qname, cs=None, ops=None, cigar=None, md=None,
            refseq=None):
        """the record's ops come from `ops`, else from `cs`, else from `cigar` + `md` (parse_md), else from `cigar` + the
        contig's `refseq` (parse_ref)"""
        qb = qseq.encode() if isinstance(qseq, str) else bytes(qseq)
        if ops is None and cs is None and md is not None:
            ops, rspan, qspan = parse_md(cigar, md, qb.decode(), qstart, qname)
        elif ops is None and cs is None and refseq is not None:
            ops, rspan, qspan = parse_ref(cigar, refseq, tstart, qb.decode(), qstart, qname)
        elif ops is None:
            ops, rspan, qspan = parse_cs(cs, qb.decode(), qstart)
        else:
            ops = [int(w) for w in ops]
            rspan = sum((w >> 2) if (w & 3) in (abi.OP_MATCH, abi.OP_DEL) else (1 if (w & 3) == abi.OP_SUB else 0) for w in ops)
            qspan = sum((w >> 2) if (w & 3) in (abi.OP_MATCH, abi.OP_INS) else (1 if (w & 3) == abi.OP_SUB else 0) for w in ops)
        if tend is not None and rspan != tend - tstart:
            raise BatchFormatError("%s: cs reference span %d != CIGAR span %d" % (qname, rspan, tend - tstart))
        if qend is not None and qspan != qend - qstart:
            raise BatchFormatError("%s: cs query span %d != aligned query span %d" % (qname, qspan, qend - qstart))
        if bq is None or len(bq) != len(qb):
            raise BatchFormatError("%s: base qualities missing or of the wrong length" % qname)
        packed = pack_seq(qb, ops, qstart)
        c = self.cols
        c["tstart"].append(tstart); c["tend"].append(tstart + rspan); c["qstart"].append(qstart)
        c["qlen"].append(len(qb)); c["mapq"].append(mapq)
        c["flags"].append(abi.READ_SECONDARY if is_secondary else 0)
        c["qname_id"].append(self.qnames.setdefault(qname, len(self.qnames)))
        c["seq_off"].append(self.seq_n); c["bq_off"].append(self.bq_n); c["op_off"].append(self.ops_n)
        c["n_ops"].append(len(ops))
        sp = np.pad(packed, (0, (-packed.size) % 16))
        bp = np.pad(np.frombuffer(bytes(bq), dtype=np.uint8), (0, (-len(qb)) % 16))
        self.seq.append(sp); self.bq.append(bp); self.ops.append(np.asarray(ops, dtype=np.uint32))
        self.seq_n += sp.size; self.bq_n += bp.size; self.ops_n += len(ops)

    def finish(self):
        cat = lambda parts, dt: (np.concatenate(parts).astype(dt) if parts else np.zeros(0, dt))
        seq, bq = cat(self.seq, np.uint8), cat(self.bq, np.uint8)
        if seq.size == 0:
            seq = np.zeros(16, np.uint8)
        if bq.size == 0:
            bq = np.zeros(16, np.uint8)
        ts = np.asarray(self.cols["tstart"], np.int32)
        if ts.size > 1 and (np.diff(ts) < 0).any():
            raise BatchFormatError("records are not coordinate sorted")
        return abi.ReadBatch(seq=seq, bq=bq, ops=cat(self.ops, np.uint32), **self.cols)
