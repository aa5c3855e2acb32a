"""Records without cs:Z decoded from CIGAR + MD:Z: pack.parse_md (the specification) against the cs ops of the same
alignment, the native host decoder against the specification byte for byte, the cs / MD / MD_EQX writer forms of one
batch to the same batch, and the rejections of the MD path in both implementations with the same words."""
import numpy as np
import pytest

import cases
import test_bamdec as tb
from himut_b200 import abi, bamdec, bamio, bamlib, pack, synth

M, I, D, S, H, EQ, X = 0, 1, 2, 4, 5, 7, 8
MATCH = lambda n: abi.make_op(abi.OP_MATCH, n)
SUB = lambda r, a: abi.make_sub(abi.BASE2CODE.get(r, abi.BASE_N), abi.BASE2CODE[a])
INS = lambda n: abi.make_op(abi.OP_INS, n)
DEL = lambda n: abi.make_op(abi.OP_DEL, n)


# ------------------------------------------------------------------------------ parse_md KATs
def test_survey_appendix_b_kat_through_md():
    """SURVEY Appendix B's cs KAT as CIGAR + MD.  cs takes a SUB's alt base from the tag, MD from SEQ: query 6 is G
    here (Appendix B's read has A there, where cs says g) so that the two describe the same alignment."""
    read = "NNACGTGCGTTTGACCA"
    want, rspan, qspan = pack.parse_cs(":4*ag:2+tt:1-ca:3", read, 2)
    cigar = [(S, 2), (M, 7), (I, 2), (M, 1), (D, 2), (M, 3), (S, 2)]
    got = pack.parse_md(cigar, "4A3^CA3", read, 2)
    assert got == (want, rspan, qspan)
    assert want == [MATCH(4), SUB("A", "G"), MATCH(2), INS(2), MATCH(1), DEL(2), MATCH(3)] and (rspan, qspan) == (13, 13)


def test_eqx_cigar_gives_the_m_cigar_ops():
    read = "NNACGTGCGTTTGACCA"
    m = pack.parse_md([(S, 2), (M, 7), (I, 2), (M, 1), (D, 2), (M, 3), (S, 2)], "4A3^CA3", read, 2)
    eqx = pack.parse_md([(S, 2), (EQ, 4), (X, 1), (EQ, 2), (I, 2), (EQ, 1), (D, 2), (EQ, 3), (S, 2)], "4A3^CA3", read, 2)
    assert eqx == m
    # a match run goes on across = / M boundaries and across MD numbers
    assert pack.parse_md([(EQ, 3), (M, 2), (EQ, 1)], "6", "ACGTAC", 0)[0] == [MATCH(6)]


def test_md_zero_separators_and_n_reference_letters():
    # a deletion at the start, adjacent SUBs, a SUB at the very end, trailing 0
    got = pack.parse_md([(D, 2), (M, 6)], "0^NN1A0C3", "GTACGT", 0)[0]
    assert got == [DEL(2), MATCH(1), SUB("A", "T"), SUB("C", "A"), MATCH(3)]
    got = pack.parse_md([(M, 4)], "1N1G0", "ACGT", 0)[0]  # an N reference letter, a SUB at the very end
    assert got == [MATCH(1), abi.make_sub(abi.BASE_N, abi.BASE2CODE["C"]), MATCH(1), SUB("G", "T")]
    # lower-case and IUPAC letters: outside ACGT -> N, as cs "*nx"
    assert pack.parse_md([(M, 3)], "1r1", "ACG", 0)[0] == [MATCH(1), abi.make_sub(abi.BASE_N, abi.BASE2CODE["C"]), MATCH(1)]
    assert pack.parse_md([(M, 3)], "1t1", "ACG", 0)[0] == [MATCH(1), SUB("T", "C"), MATCH(1)]
    # a SUB whose alt equals the MD letter is still a SUB (cs "*aa" is not checked either)
    assert pack.parse_md([(M, 1)], "0A0", "A", 0)[0] == [SUB("A", "A")]
    # insertions split match runs; MD skips them
    assert pack.parse_md([(M, 2), (I, 3), (M, 2)], "4", "ACGGGTA", 0)[0] == [MATCH(2), INS(3), MATCH(2)]
    # zero-length ops are skipped
    assert pack.parse_md([(M, 2), (I, 0), (M, 2)], "4", "ACGT", 0)[0] == [MATCH(4)]


@pytest.mark.parametrize("cigar, md, seq, key, arg", [
    ([(M, 4)], "4x", "ACGT", "md_token", 1),
    ([(M, 4)], "", "ACGT", "md_token", 0),
    ([(M, 4)], "A3", "ACGT", "md_token", 0),
    ([(M, 4)], "2^3", "ACGT", "md_token", 1),
    ([(M, 4)], "2A1^", "ACGT", "md_token", 3),
    ([(EQ, 4)], "2A1", "ACGT", "md_span", 2),            # = over an MD mismatch
    ([(X, 1), (M, 3)], "4", "ACGT", "md_span", 0),       # X over an MD match
    ([(M, 4)], "3", "ACGT", "md_span", 3),               # MD runs out
    ([(M, 4)], "5", "ACGT", "md_span", 4),               # MD left over
    ([(M, 4)], "4A0", "ACGT", "md_span", 4),
    ([(M, 2), (D, 2), (M, 2)], "2^A2", "ACGT", "md_span", 2),   # D longer than its ^ letters
    ([(M, 2), (D, 1), (M, 2)], "3^A1", "ACGT", "md_span", 2),   # D where MD has a match
    ([(M, 4)], "2^A2", "ACGT", "md_span", 2),            # ^ where the CIGAR has M
    ([(M, 2), (3, 5), (M, 2)], "4", "ACGT", "cigar_op", 1),     # N
    ([(M, 2), (6, 1), (M, 2)], "4", "ACGT", "cigar_op", 1),     # P
    ([(M, 2), (S, 1), (M, 1)], "3", "ACGT", "cigar_op", 1),     # a soft clip inside
    ([(M, 2), (H, 1), (M, 2)], "4", "ACGT", "cigar_op", 1),     # a hard clip inside
    ([(M, 5)], "5", "ACGT", "span_qry", 5),              # CIGAR query length != SEQ length
    ([(M, 4)], "4", "ACNT", "n_match", 2),
    ([(M, 4)], "2G1", "ACNT", "sub_n", 2),
])
def test_parse_md_rejections(cigar, md, seq, key, arg):
    with pytest.raises(pack.BatchFormatError) as ex:
        pack.parse_md(cigar, md, seq, 0, "q")
    assert str(ex.value) == pack.MD_ERR[key] % ("q", arg)


# ------------------------------------------------------------------------------ native decoder = specification
WINDOWS = [(0, 300_000), (1, 200_000), (200_000, 299_998), (123_456, 123_457), (299_990, 300_000), (0, 1)]


@pytest.mark.parametrize("writer", ["python", "native"])
@pytest.mark.parametrize("tags", ["md", "md_eqx"])
@pytest.mark.parametrize("threads", [1, 4])
def test_native_md_batch_equals_python_batch(tmp_path, writer, tags, threads):
    d = synth.generate(300_000, seed=11)
    path = str(tmp_path / "t.bam")
    (bamio.write_batch_bam if writer == "python" else bamdec.write_batch_bam)(path, "chr1", 300_000, d.batch, tags=tags)
    rd = bamio.BamReader(path)
    r0 = next(rd.fetch("chr1"))
    assert "MD" in r0.tags and "cs" not in r0.tags
    nb = bamdec.NativeBam(path, threads=threads)
    qnames = {}
    for s, e in WINDOWS:
        bb = pack.BatchBuilder()
        bb.qnames = qnames
        tb._same(nb.read_batch("chr1", s, e), bamio.read_batch(rd, "chr1", s, e, builder=bb))
    assert cases.batch_digest(nb.read_batch("chr1", 0, 300_000)) == cases.batch_digest(d.batch)
    nb.close(); rd.close()


def test_native_md_writer_equals_python_writer(tmp_path):
    d = synth.generate(150_000, seed=14)
    for tags in ("md", "md_eqx"):
        p_py, p_c = str(tmp_path / ("py_%s.bam" % tags)), str(tmp_path / ("c_%s.bam" % tags))
        bamio.write_batch_bam(p_py, "chr1", 150_000, d.batch, tags=tags)
        bamdec.write_batch_bam(p_c, "chr1", 150_000, d.batch, threads=3, tags=tags)
        key = lambda r: (r.query_name, r.reference_start, r.cigar, r.tags.get("MD"), r.tags.get("cs"), r.tags.get("tp"),
                         bytes(r.qual), bytes(r.seq_nibbles))
        a, b = bamio.BamReader(p_py), bamio.BamReader(p_c)
        assert [key(r) for r in a.fetch("chr1")] == [key(r) for r in b.fetch("chr1")]
    with pytest.raises(ValueError):
        bamdec.write_batch_bam(p_c, "chr1", 150_000, d.batch, tags="MD")


def _decode_all(path, seq=True, compact=False, threads=2):
    nb = bamdec.NativeBam(path, threads=threads)
    try:
        out = nb.read_batch("chr1", 0, nb.lengths[0], seq=seq, compact=compact)
        if compact:
            b, cq = out
            return cases.batch_digest(b), (cq.mask.tobytes(), cq.exc[:cq.n_exc].tobytes(), cq.exc_off.tobytes(), cq.modal)
        return cases.batch_digest(out), None
    finally:
        nb.close()


def test_synth_ops_agree_with_seq():
    """the comparisons below rely on it: in synth.generate's batches the alt base of every SUB is the read base at its
    query position (MD takes the alt from SEQ, cs from the op) and no two MATCH ops are adjacent"""
    for seed in (1, 2):
        b = synth.generate(120_000, seed=seed).batch
        assert _canonical(b) is b


@pytest.mark.parametrize("seed, n", [(1, 60_000), (2, 250_000), (3, 400_000)])
def test_three_writer_forms_decode_to_one_batch(tmp_path, seed, n):
    d = synth.generate(n, seed=seed)
    paths = {}
    for tags in ("cs", "md", "md_eqx"):
        paths[tags] = str(tmp_path / ("%s.bam" % tags))
        bamdec.write_batch_bam(paths[tags], "chr1", n, d.batch, tags=tags)
    for seq, compact in ((True, False), (False, False), (False, True)):
        want = _decode_all(paths["cs"], seq, compact)
        for tags in ("md", "md_eqx"):
            assert _decode_all(paths[tags], seq, compact) == want, (tags, seq, compact)


def test_mixed_cs_and_md_records(tmp_path):
    """a BAM whose records alternate between cs:Z and MD:Z decodes to the all-cs batch, natively and in Python"""
    n = 200_000
    d = synth.generate(n, seed=7)
    p_cs, p_md, p_mix = (str(tmp_path / x) for x in ("cs.bam", "md.bam", "mix.bam"))
    bamio.write_batch_bam(p_cs, "chr1", n, d.batch)
    bamio.write_batch_bam(p_md, "chr1", n, d.batch, tags="md")
    a, b = list(bamio.BamReader(p_cs).fetch("chr1")), list(bamio.BamReader(p_md).fetch("chr1"))
    w = bamio.BamWriter(p_mix, [("chr1", n)])
    for i, (x, y) in enumerate(zip(a, b)):
        r = x if i % 2 else y
        w.add(r.ref_id, r.reference_start, r.query_name, r.flag, r.mapping_quality, r.cigar, r.query_sequence, bytes(r.qual),
              [(t, "A" if t == "tp" else "Z", v) for t, v in r.tags.items()])
    w.close()
    want = cases.batch_digest(bamdec.NativeBam(p_cs).read_batch("chr1", 0, n))
    assert cases.batch_digest(bamdec.NativeBam(p_mix, threads=3).read_batch("chr1", 0, n)) == want
    assert cases.batch_digest(bamio.read_batch(bamio.BamReader(p_mix), "chr1", 0, n)) == want


def _canonical(batch):
    """the batch with adjacent MATCH ops merged and each SUB's alt set to the read base at its query position (the
    batch itself when nothing changes).  MD cannot say where one match block ends and the next begins, and the cs
    writer keeps the blocks apart, so an op stream with adjacent MATCH ops reads back merged from MD only — and
    normcounts evaluates its mismatch window once per match block, so the split is not cosmetic.  The alt rewrite
    matters for generators whose SUB ops disagree with SEQ: cs carries the op's alt, MD the read's base."""
    bb = pack.BatchBuilder()
    changed = False
    for r in range(batch.n_reads):
        so, oo, ql = int(batch.seq_off[r]), int(batch.op_off[r]), int(batch.qlen[r])
        codes = ((batch.seq[so:so + (ql + 3) // 4][:, None] >> np.array([0, 2, 4, 6], np.uint8)) & 3).reshape(-1)[:ql]
        ops, q = [], int(batch.qstart[r])
        for w in batch.ops[oo:oo + int(batch.n_ops[r])]:
            kind, val = int(w) & 3, int(w) >> 2
            if kind == abi.OP_MATCH and ops and ops[-1] & 3 == abi.OP_MATCH:
                ops[-1] = abi.make_op(abi.OP_MATCH, (ops[-1] >> 2) + val); changed = True
            elif kind == abi.OP_SUB:
                fixed = abi.make_sub(val & 7, int(codes[q]))
                changed |= fixed != int(w)
                ops.append(fixed)
            else:
                ops.append(int(w))
            q += val if kind in (abi.OP_MATCH, abi.OP_INS) else (1 if kind == abi.OP_SUB else 0)
        bb.add(tstart=int(batch.tstart[r]), tend=None, qstart=int(batch.qstart[r]), qend=None,
               qseq="".join("ATGC"[c] for c in codes), bq=batch.bq[int(batch.bq_off[r]):int(batch.bq_off[r]) + ql].tobytes(),
               mapq=int(batch.mapq[r]), is_secondary=bool(batch.flags[r] & abi.READ_SECONDARY),
               qname="read%d" % int(batch.qname_id[r]), ops=ops)
    return bb.finish() if changed else batch


@pytest.mark.parametrize("seed", [1, 2, 5])
def test_adversarial_md_equals_cs_of_the_canonical_ops(tmp_path, seed):
    batch, _ref = cases.adversarial_batch(seed, contig_len=6000, n_reads=300, max_len=2000)
    canon = _canonical(batch)
    p_cs, p_md, p_eqx = (str(tmp_path / x) for x in ("cs.bam", "md.bam", "eqx.bam"))
    bamio.write_batch_bam(p_cs, "chr1", 6000, canon)
    bamio.write_batch_bam(p_md, "chr1", 6000, batch, tags="md")
    bamdec.write_batch_bam(p_eqx, "chr1", 6000, batch, tags="md_eqx")
    want = _decode_all(p_cs)
    assert _decode_all(p_md) == want and _decode_all(p_eqx, threads=1) == want
    assert cases.batch_digest(bamio.read_batch(bamio.BamReader(p_md), "chr1", 0, 6000)) == want[0]


# ------------------------------------------------------------------------------ rejections
def _md_rec(cigar=((M, 8),), md="8", seq="ACGTACGT", **k):
    return tb._rec(cigar=cigar, seq=seq, cs=None, extra=[("MD", "Z", md)], **k)


MD_BAD = [
    (dict(md="8x"), "md_token", 1),
    (dict(md="3A3"), "md_span", 7),
    (dict(cigar=((EQ, 3), (X, 1), (EQ, 4)), md="8"), "md_span", 3),
    (dict(cigar=((EQ, 8),), md="3G4"), "md_span", 3),
    (dict(cigar=((M, 4), (D, 2), (M, 4)), md="4^A4"), "md_span", 4),
    (dict(cigar=((M, 4), (3, 100), (M, 4)), md="8"), "cigar_op", 1),
    (dict(cigar=((M, 4), (6, 2), (M, 4)), md="8"), "cigar_op", 1),
    (dict(cigar=((M, 4), (S, 1), (M, 3)), md="7"), "cigar_op", 1),
    (dict(cigar=((M, 9),), md="9"), "span_qry", 9),
    (dict(seq="ACNTACGT"), "n_match", 2),
    (dict(seq="ACNTACGT", md="2G5"), "sub_n", 2),
]


@pytest.mark.parametrize("bad, key, arg", MD_BAD)
def test_md_rejections_have_the_same_words_in_both_implementations(tmp_path, bad, key, arg):
    path = str(tmp_path / "b.bam")
    tb._write(path, [_md_rec(qname="mdrec", **bad)])
    want = pack.MD_ERR[key] % ("mdrec", arg)
    nb = bamdec.NativeBam(path, threads=1)
    for seq in (True, False):
        with pytest.raises(pack.BatchFormatError) as ex:
            nb.read_batch("chr1", 0, 1000, seq=seq)
        assert str(ex.value) == want
    with pytest.raises(pack.BatchFormatError) as ex:
        bamio.read_batch(bamio.BamReader(path), "chr1", 0, 1000)
    assert str(ex.value) == want


def test_neither_tag_is_still_no_cs(tmp_path):
    path = str(tmp_path / "n.bam")
    tb._write(path, [tb._rec(cs=None, qname="bare")])
    for read in (lambda: bamdec.NativeBam(path, threads=1).read_batch("chr1", 0, 1000),
                 lambda: bamio.read_batch(bamio.BamReader(path), "chr1", 0, 1000)):
        with pytest.raises(pack.BatchFormatError) as ex:
            read()
        assert str(ex.value).startswith("bare has no cs:Z tag (the reference raises KeyError in BAM.__init__)")


def test_cs_wins_over_md(tmp_path):
    """a record with both tags is decoded from cs, exactly as before: a wrong MD next to it changes nothing"""
    path, plain = str(tmp_path / "both.bam"), str(tmp_path / "cs.bam")
    tb._write(path, [tb._rec(cs=":3*ag:4", seq="ACGGACGT", extra=[("MD", "Z", "garbage")])])
    tb._write(plain, [tb._rec(cs=":3*ag:4", seq="ACGGACGT")])
    want = cases.batch_digest(bamdec.NativeBam(plain).read_batch("chr1", 0, 1000))
    assert cases.batch_digest(bamdec.NativeBam(path).read_batch("chr1", 0, 1000)) == want
    assert cases.batch_digest(bamio.read_batch(bamio.BamReader(path), "chr1", 0, 1000)) == want


def test_window_qlens_and_thresholds_on_md(tmp_path):
    n = 300_000
    d = synth.generate(n, seed=19)
    p_cs, p_md = str(tmp_path / "cs.bam"), str(tmp_path / "md.bam")
    bamdec.write_batch_bam(p_cs, "chr1", n, d.batch)
    bamdec.write_batch_bam(p_md, "chr1", n, d.batch, tags="md")
    a, b = bamdec.NativeBam(p_cs), bamdec.NativeBam(p_md)
    for s, e in ((0, n), (100_000, 200_000), (5, 6)):
        assert np.array_equal(a.window_qlens("chr1", s, e), b.window_qlens("chr1", s, e))
    tsize = {"chr1": n}
    assert bamlib.get_thresholds(p_cs, ["chr1"], tsize) == bamlib.get_thresholds(p_md, ["chr1"], tsize)
