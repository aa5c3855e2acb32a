"""Records with neither cs:Z nor MD:Z decoded from CIGAR + the reference FASTA: pack.parse_ref (the specification)
against the cs ops of the same alignment, the native host decoder against the specification byte for byte, the cs /
eqx / m writer forms of one batch to the same batch, the rejections of the reference path in both implementations
with the same words, fasta.py, and the drop-in `call` worker reading its FASTA from HIMUT_B200_REF."""
import gzip
import os

import pytest

import cases
import parity
import test_bamdec as tb
import test_md_ops as tm
import test_worker_host as tw
from test_worker_host import octx  # noqa: F401  (the oracle stand-in context, a fixture)
from himut_b200 import abi, bamdec, bamio, fasta, pack, synth

M, I, D, S, H, EQ, X = 0, 1, 2, 4, 5, 7, 8
MATCH, SUB, INS, DEL = tm.MATCH, tm.SUB, tm.INS, tm.DEL


def write_fasta(path, contigs, width=60):
    """[(name, seq bytes / str, header suffix)] -> FASTA with lines of `width` bases"""
    with open(path, "w") as f:
        for name, seq, extra in contigs:
            seq = seq.decode() if isinstance(seq, bytes) else seq
            f.write(">%s%s\n" % (name, extra) + "".join(seq[i:i + width] + "\n" for i in range(0, len(seq), width)))


# ------------------------------------------------------------------------------ parse_ref KATs (each = parse_cs)
REF = "GGACGTACGTNNACGTRYacgtACGTACGTAC"


@pytest.mark.parametrize("cigar, tstart, read, qstart, cs", [
    # M with mismatches at the first and the last aligned base, and two adjacent ones
    ([(M, 8)], 2, "TCGTACGA", 0, "*at:6*ta"),
    ([(M, 8)], 2, "ACCAACGT", 0, ":2*gc*ta:4"),
    # reference N and an IUPAC letter under M and X: SUB(N, read base)
    ([(M, 8)], 8, "GTGCACGT", 0, ":2*ng*nc:4"),
    ([(EQ, 2), (X, 2), (EQ, 2)], 14, "GTACAC", 0, ":2*ra*yc:2"),
    # lower-case reference
    ([(M, 6)], 18, "ACCTAC", 0, ":2*gc:3"),
    # =/X runs merge with M runs; I / D next to mismatches
    ([(EQ, 2), (M, 2), (X, 1), (M, 3)], 2, "ACGTTCGT", 0, ":4*at:3"),
    ([(M, 3), (I, 2), (X, 1), (D, 2), (EQ, 2)], 2, "ACGTTGGT", 0, ":3+tt*tg-ac:2"),
    ([(D, 1), (X, 1), (I, 1), (M, 4)], 2, "TCGTAC", 0, "-a*ct+c:4"),
    # soft and hard clips, ops of length 0
    ([(H, 5), (S, 2), (M, 4), (S, 1), (H, 3)], 2, "NNACGTN", 2, ":4"),
    ([(S, 1), (M, 2), (I, 0), (M, 2), (D, 0), (EQ, 0), (M, 2)], 2, "TACGTAC", 1, ":6"),
])
def test_parse_ref_kats_equal_parse_cs(cigar, tstart, read, qstart, cs):
    want = pack.parse_cs(cs, read, qstart)
    assert pack.parse_ref(cigar, REF, tstart, read, qstart) == want
    assert pack.parse_ref(cigar, REF.encode(), tstart, read, qstart) == want


def test_parse_ref_spells_out_the_ops():
    assert pack.parse_ref([(M, 8)], REF, 2, "TCGTACGA", 0)[0] == [SUB("A", "T"), MATCH(6), SUB("T", "A")]
    assert pack.parse_ref([(M, 3)], REF, 9, "TAC", 0)[0] == [MATCH(1), abi.make_sub(abi.BASE_N, 0), abi.make_sub(abi.BASE_N, 3)]
    assert pack.parse_ref([(M, 4), (I, 1), (M, 4)], REF, 2, "ACGTAACGT", 0) == ([MATCH(4), INS(1), MATCH(4)], 8, 9)


@pytest.mark.parametrize("cigar, tstart, read, key, arg", [
    ([(EQ, 4)], 2, "ACCT", "ref_span", 2),                # = over a mismatch
    ([(EQ, 2), (EQ, 2)], 8, "GTAC", "ref_span", 2),       # = over a reference N
    ([(X, 1), (M, 3)], 2, "ACGT", "ref_span", 0),         # X over a match
    ([(M, 4)], 2, "ACNT", "sub_n", 2),                    # read N under M (even where it matches nothing)
    ([(EQ, 4)], 2, "ACNT", "n_match", 2),                 # read N under =
    ([(X, 2)], 2, "TN", "sub_n", 1),                      # read N under X
    ([(M, 4)], len(REF) - 3, "ACGT", "ref_end", len(REF) + 1),   # past the end of the reference
    ([(M, 2), (D, 4)], len(REF) - 4, "AC", "ref_end", len(REF) + 2),
    ([(M, 2), (3, 5), (M, 2)], 2, "ACGT", "cigar_op", 1),  # N
    ([(M, 2), (S, 1), (M, 1)], 2, "ACGT", "cigar_op", 1),  # a soft clip inside
    ([(M, 5)], 2, "ACGT", "span_qry", 5),
])
def test_parse_ref_rejections(cigar, tstart, read, key, arg):
    with pytest.raises(pack.BatchFormatError) as ex:
        pack.parse_ref(cigar, REF, tstart, read, 0, "q")
    assert str(ex.value) == (pack.REF_ERR.get(key) or pack.MD_ERR[key]) % ("q", arg)


def test_past_the_end_is_checked_before_any_base():
    """a bad read base inside an alignment that also runs past the end: the bounds check comes first"""
    with pytest.raises(pack.BatchFormatError, match="past the end"):
        pack.parse_ref([(M, 6)], "ACGT", 0, "NNNNNN", 0, "q")


# ------------------------------------------------------------------------------ writer forms, native = specification
def _paths(tmp_path, n, batch, forms=("cs", "eqx", "m"), writer="native"):
    out = {}
    for tags in forms:
        out[tags] = str(tmp_path / ("%s_%s.bam" % (writer, tags)))
        (bamdec.write_batch_bam if writer == "native" else bamio.write_batch_bam)(out[tags], "chr1", n, batch, tags=tags)
    return out


def _decode(path, ref, seq=True, compact=False, threads=2):
    nb = bamdec.NativeBam(path, threads=threads)
    try:
        nb.set_reference("chr1", ref)
        out = nb.read_batch("chr1", 0, nb.lengths[0], seq=seq, compact=compact)
        if compact:
            b, cq = out
            return cases.batch_digest(b), (cq.mask.tobytes(), cq.exc[:cq.n_exc].tobytes(), cq.exc_off.tobytes(), cq.modal)
        return cases.batch_digest(out), None
    finally:
        nb.close()


@pytest.mark.parametrize("writer", ["python", "native"])
@pytest.mark.parametrize("seed, n", [(1, 60_000), (3, 250_000)])
def test_writer_forms_decode_to_the_cs_batch(tmp_path, writer, seed, n):
    d = synth.generate(n, seed=seed)
    paths = _paths(tmp_path, n, d.batch, writer=writer)
    for seq, compact in ((True, False), (False, False), (False, True)):
        want = tm._decode_all(paths["cs"], seq, compact)
        for tags in ("eqx", "m"):
            for threads in (1, 4):
                assert _decode(paths[tags], d.ref, seq, compact, threads) == want, (tags, seq, compact, threads)


@pytest.mark.parametrize("tags", ["eqx", "m"])
def test_native_equals_the_specification(tmp_path, tags):
    n = 300_000
    d = synth.generate(n, seed=11)
    path = _paths(tmp_path, n, d.batch, forms=(tags,))[tags]
    rd = bamio.BamReader(path)
    r0 = next(rd.fetch("chr1"))
    assert "MD" not in r0.tags and "cs" not in r0.tags
    nb = bamdec.NativeBam(path, threads=3)
    nb.set_reference("chr1", d.ref.decode())  # str works as bytes
    qnames = {}
    for s, e in tm.WINDOWS:
        bb = pack.BatchBuilder()
        bb.qnames = qnames
        tb._same(nb.read_batch("chr1", s, e), bamio.read_batch(rd, "chr1", s, e, builder=bb, refseq=d.ref))
    assert cases.batch_digest(nb.read_batch("chr1", 0, n)) == cases.batch_digest(d.batch)
    nb.close(); rd.close()


@pytest.mark.parametrize("seed", [1, 2, 5])
def test_adversarial_forms_equal_cs(tmp_path, seed):
    """N reference letters, dense events, clips, secondary records, duplicate names"""
    batch, ref = cases.adversarial_batch(seed, contig_len=6000, n_reads=300, max_len=2000)
    canon = tm._canonical(batch)
    p_cs = str(tmp_path / "cs.bam")
    bamio.write_batch_bam(p_cs, "chr1", 6000, canon)
    want = tm._decode_all(p_cs)
    for writer in ("python", "native"):
        paths = _paths(tmp_path, 6000, batch, forms=("eqx", "m"), writer=writer)
        for tags, p in paths.items():
            assert _decode(p, ref) == want, (writer, tags)
            assert cases.batch_digest(bamio.read_batch(bamio.BamReader(p), "chr1", 0, 6000, refseq=ref)) == want[0]


def test_mixed_cs_md_and_tagless_records(tmp_path):
    n = 200_000
    d = synth.generate(n, seed=7)
    p_cs, p_mix = str(tmp_path / "cs.bam"), str(tmp_path / "mix.bam")
    forms = {t: list(bamio.BamReader(p).fetch("chr1")) for t, p in _paths(tmp_path, n, d.batch, forms=("cs", "md", "m"), writer="python").items()}
    w = bamio.BamWriter(p_mix, [("chr1", n)])
    for i, r in enumerate(zip(forms["cs"], forms["md"], forms["m"])):
        r = r[i % 3]
        w.add(r.ref_id, r.reference_start, r.query_name, r.flag, r.mapping_quality, r.cigar, r.query_sequence, bytes(r.qual),
              [(t, "A" if t == "tp" else "Z", v) for t, v in r.tags.items()])
    w.close()
    bamio.write_batch_bam(p_cs, "chr1", n, d.batch)
    want = cases.batch_digest(bamdec.NativeBam(p_cs).read_batch("chr1", 0, n))
    assert _decode(p_mix, d.ref, threads=3)[0] == want
    assert cases.batch_digest(bamio.read_batch(bamio.BamReader(p_mix), "chr1", 0, n, refseq=d.ref)) == want


def test_reference_of_another_contig_is_not_used(tmp_path):
    """only records of the contig whose sequence was set decode from it; a cs record never reads it"""
    path = str(tmp_path / "two.bam")
    tb._write(path, [tb._rec(pos=10, ref_id=1, cs=None, qname="other"), tb._rec(pos=10, cs=":8", qname="withcs")])
    nb = bamdec.NativeBam(path, threads=1)
    nb.set_reference("chr1", "N" * 1000)
    assert nb.read_batch("chr1", 0, 1000).n_reads == 1
    with pytest.raises(pack.BatchFormatError, match="^other has no cs:Z tag"):
        nb.read_batch("chr2", 0, 1000)
    nb.set_reference("chr1", None)
    nb.close()


# ------------------------------------------------------------------------------ rejections: same words
def _ref_rec(cigar=((M, 8),), seq="ACGTACGT", pos=10, **k):
    return tb._rec(pos=pos, cigar=cigar, seq=seq, cs=None, **k)


TB_REF = ("ACGT" * 250).encode()  # the 1000-base chr1 of tb._write; position 10 holds G
REF_BAD = [
    (dict(cigar=((EQ, 8),), seq="GTACGTAA"), "ref_span", 7),
    (dict(cigar=((X, 1), (EQ, 7)), seq="GTACGTAC"), "ref_span", 0),
    (dict(cigar=((M, 8),), seq="GTNCGTAC"), "sub_n", 2),
    (dict(cigar=((EQ, 8),), seq="GTNCGTAC"), "n_match", 2),
    (dict(cigar=((X, 2), (M, 6)), seq="ANACGTAC"), "sub_n", 1),
    (dict(pos=995, seq="GTACGTAC"), "ref_end", 1003),
    (dict(cigar=((M, 4), (3, 100), (M, 4))), "cigar_op", 1),
    (dict(cigar=((M, 9),)), "span_qry", 9),
    # D lengths no query length bounds: a reference span of 2^32 + 1 that an int32 sum wraps to 1
    (dict(cigar=((M, 1),) + ((D, (1 << 28) - 1),) * 16 + ((M, 16),), seq="G" + "TACG" * 4), "ref_end", 10 + (1 << 32) + 1),
]


@pytest.mark.parametrize("bad, key, arg", REF_BAD)
def test_ref_rejections_have_the_same_words_in_both_implementations(tmp_path, bad, key, arg):
    path = str(tmp_path / "b.bam")
    tb._write(path, [_ref_rec(qname="refrec", **bad)])
    want = (pack.REF_ERR.get(key) or pack.MD_ERR[key]) % ("refrec", arg)
    nb = bamdec.NativeBam(path, threads=1)
    nb.set_reference("chr1", TB_REF)
    for seq in (True, False):
        with pytest.raises(pack.BatchFormatError) as ex:
            nb.read_batch("chr1", 0, 1000, seq=seq)
        assert str(ex.value) == want
    with pytest.raises(pack.BatchFormatError) as ex:
        bamio.read_batch(bamio.BamReader(path), "chr1", 0, 1000, refseq=TB_REF)
    assert str(ex.value) == want


def test_tagless_bams_without_a_reference_are_still_no_cs(tmp_path):
    d = synth.generate(60_000, seed=2)
    for tags, p in _paths(tmp_path, 60_000, d.batch, forms=("eqx", "m")).items():
        for read in (lambda: bamdec.NativeBam(p, threads=1).read_batch("chr1", 0, 60_000),
                     lambda: bamio.read_batch(bamio.BamReader(p), "chr1", 0, 60_000)):
            with pytest.raises(pack.BatchFormatError) as ex:
                read()
            assert str(ex.value).startswith("read0 has no cs:Z tag (the reference raises KeyError in BAM.__init__)"), tags


def test_reference_length_and_contig_are_checked(tmp_path):
    path = str(tmp_path / "b.bam")
    tb._write(path, [_ref_rec()])
    nb = bamdec.NativeBam(path, threads=1)
    with pytest.raises(pack.BatchFormatError) as ex:
        nb.set_reference("chr1", TB_REF[:999])
    assert str(ex.value) == "the reference sequence of chr1 has 999 bases, its @SQ LN 1000"
    with pytest.raises(pack.BatchFormatError, match="no cs:Z tag"):  # a rejected reference is not kept
        nb.read_batch("chr1", 0, 1000)
    fa = str(tmp_path / "r.fa")
    write_fasta(fa, [("chr1", TB_REF[:999], "")])
    with pytest.raises(ValueError) as ex:
        fasta.load_contig(fa, "chr1", 1000)
    assert "999 bases" in str(ex.value) and "1000" in str(ex.value) and fa in str(ex.value)
    with pytest.raises(ValueError) as ex:
        fasta.load_contig(fa, "chr2")
    assert str(ex.value) == "contig chr2 is not in the FASTA %s" % fa


# ------------------------------------------------------------------------------ fasta.py
def test_fasta_wrapped_lines_fai_and_scan_agree(tmp_path):
    seqs = [("chrA", "ACGTN" * 37 + "acg", " some description"), ("chr1", TB_REF.decode(), ""), ("chrE", "", ""),
            ("chrZ", "acgtRYKM" * 20, "\tLN:160")]
    for width in (7, 60, 1000):
        fa = str(tmp_path / ("w%d.fa" % width))
        write_fasta(fa, seqs, width)
        scanned = {n: fasta.load_contig(fa, n) for n, _s, _e in seqs}
        assert scanned == {n: s.encode() for n, s, _e in seqs}  # header's first word, case kept, line breaks dropped
        with open(fa + ".fai", "w") as f:  # samtools faidx layout
            off = 0
            for n, s, e in seqs:
                off += len(">%s%s\n" % (n, e))
                f.write("%s\t%d\t%d\t%d\t%d\n" % (n, len(s), off, width, width + 1))
                off += len(s) + -(-len(s) // width)
        assert {n: fasta.load_contig(fa, n, len(s)) for n, s, _e in seqs} == scanned
        os.remove(fa + ".fai")
    crlf = str(tmp_path / "crlf.fa")
    open(crlf, "wb").write(b">c1 x\r\nACG\r\nTA\r\n>c2\r\nGG\r\n")
    assert fasta.load_contig(crlf, "c1") == b"ACGTA" and fasta.load_contig(crlf, "c2") == b"GG"


def test_fasta_gzip_is_rejected(tmp_path):
    fa = str(tmp_path / "r.fa.gz")
    with gzip.open(fa, "wt") as f:
        f.write(">chr1\nACGT\n")
    with pytest.raises(ValueError, match="decompress"):
        fasta.load_contig(fa, "chr1")


# ------------------------------------------------------------------------------ drop-in call worker, HIMUT_B200_REF
def test_call_worker_reads_its_fasta_from_the_environment(octx, tmp_path, monkeypatch):
    c = cases.build_case("call_config0_1mb")
    fx = parity.load_golden("call_config0_1mb")
    fa = str(tmp_path / "ref.fa")
    write_fasta(fa, [(cases.CHROM, c["ref"], "")])
    real = bamio.write_batch_bam
    monkeypatch.setattr(bamio, "write_batch_bam", lambda *a, **k: real(*a, **dict(k, tags="m")))
    monkeypatch.setenv("HIMUT_B200_REF", fa)
    rows, log = tw._run_call(c, tmp_path)
    gold = parity.golden_rows(fx)
    assert parity.rows_equal(rows, gold), parity.first_diff(rows, gold)
    assert log == fx["expected"]["log"]
    monkeypatch.delenv("HIMUT_B200_REF")
    with pytest.raises(pack.BatchFormatError, match="no cs:Z tag"):
        tw._run_call(c, tmp_path)

