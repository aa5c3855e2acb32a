"""The fp64 genotype sums on columns where the order of the additions decides the call (DESIGN.md §4, exactness rules).

The reference adds, per allele, the reads' per-BQ terms left to right in file order, then the alleles in the order
A, T, G, C from 0.0, then the prior, and multiplies by -10 (`gt_pl` in oracle/himut_oracle.c, `gt_pl_dev` in
kernels.cuh); GQ = int(second - best) capped at 99, and the tie flag is `second == best`.  On ordinary pileups a PL
summed in another order differs in the last bit or two and nothing observable moves, so this file builds columns
where it does: for every column the log10 prior of one genotype state is tuned, double by double, until the
reference-order result sits on a boundary (GQ at an integer, two PL equal, the best genotype about to change), and
kept only if some plausible kernel mistake lands on the other side of it.

CPU: a plain restatement of the model (pinned to the oracle on every column), the mistake evaluators, the proof
that the set is not vacuous, and the soundness of the normcounts certificate (DESIGN.md §4.1) against the
restatement.  GPU: every column through every `call` and `normcounts` route against the oracle, and pure columns at
the certificate's edge through the bit path.
"""
import functools
import math
import operator
import random
from fractions import Fraction

import numpy as np
import pytest

import cases
import parity
import test_norm_cert
from himut_b200 import abi, gtmodel, pack
from oracle import oracle

# ---------------------------------------------------------------- the genotype model, restated ------------------
GT_B1 = (0, 1, 3, 2, 1, 3, 2, 3, 2, 2)  # gtlib.gt_lst as base codes A0 T1 G2 C3
GT_B2 = (0, 0, 0, 0, 1, 1, 1, 3, 3, 2)
BASES = "ATGC"
ATGC = (0, 1, 2, 3)
HOMREF, HET, HETALT, HOMALT = 0, 1, 2, 3


def gt_state(b1, b2, ref):
    if b1 == ref and b2 == ref:
        return HOMREF
    if (b1 == ref) != (b2 == ref):
        return HET
    return HETALT if b1 != b2 else HOMALT


def gt_kind(g, base):
    """which per-BQ table genotype g takes for reads of `base`: 0 hom, 1 het, 2 error"""
    b1, b2 = GT_B1[g], GT_B2[g]
    if b1 == b2 and base == b1:
        return 0
    if b1 != b2 and base in (b1, b2):
        return 1
    return 2


@functools.lru_cache(maxsize=None)
def tables():
    p = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
    return tuple(tuple(t) for t in (p.lut_hom, p.lut_het, p.lut_err))


# how the reads of one allele are added.  Not sum(): since Python 3.12 it compensates float sums.
def sum_in_order(xs):
    return functools.reduce(operator.add, xs, 0.0)


def sum_reversed(xs):
    return functools.reduce(operator.add, reversed(xs), 0.0)


def sum_pairwise(xs):
    if len(xs) <= 1:
        return xs[0] if xs else 0.0
    h = len(xs) // 2
    return sum_pairwise(xs[:h]) + sum_pairwise(xs[h:])


def sum_exact(xs):
    return functools.reduce(operator.add, (Fraction(x) for x in xs), Fraction(0))


# name -> (sum of one allele's reads, allele order, exact arithmetic rounded once at the end)
EVALUATORS = {
    "reference": (sum_in_order, ATGC, False),
    "reads_reversed": (sum_reversed, ATGC, False),
    "reads_pairwise": (sum_pairwise, ATGC, False),
    "alleles_CGTA": (sum_in_order, (3, 2, 1, 0), False),
    "exact": (sum_exact, ATGC, True),
}
MISTAKES = [k for k in EVALUATORS if k != "reference"]


def allele_lists(alleles, quals):
    """per-allele BQ lists in file order (what `update_allelecounts` appends)"""
    lists = ([], [], [], [])
    for a, q in zip(alleles, quals):
        lists[BASES.index(a)].append(q)
    return lists


@functools.lru_cache(maxsize=None)
def allele_sums(quals, how):
    """(hom, het, error) sums of one allele's reads under one evaluator (quals: tuple in file order)"""
    tabs = tables()
    return tuple(EVALUATORS[how][0]([tabs[k][q] for q in quals]) for k in range(3))


def gt_pl(lists, lp, ref, skip=-1, how="reference"):
    """the ten PL of `gt_pl` (oracle) under one evaluator; skip >= 0 leaves that allele out (normcounts' second GQ)"""
    _, order, exact = EVALUATORS[how]
    S = [allele_sums(tuple(lists[a]), how) for a in range(4)]
    pl = []
    for g in range(10):
        acc = Fraction(0) if exact else 0.0
        for base in order:
            if base != skip:
                acc = acc + S[base][gt_kind(g, base)]
        prior = lp[gt_state(GT_B1[g], GT_B2[g], ref)]
        pl.append(float(-10 * (acc + Fraction(prior))) if exact else -10.0 * (acc + prior))
    return pl


def argmin_gt(pl):
    """-> (best, gq, tie): stable argmin, GQ = int(second - best) capped at 99"""
    best = 0
    for g in range(1, 10):
        if pl[g] < pl[best]:
            best = g
    second = min(pl[g] for g in range(10) if g != best)
    d = second - pl[best]
    return best, (int(d) if d < 99.0 else 99), second == pl[best]


def norm_alt(lists, ref):
    """normcounts' alt: the most frequent other allele, the first in A, T, G, C order on a tie"""
    alt = None
    for a in ATGC:
        if a != ref and (alt is None or len(lists[a]) > len(lists[alt])):
            alt = a
    return alt


def call_view(lists, lp, ref, how="reference"):
    """what a `call` record shows of the genotype: (best genotype, GQ, tie flag)"""
    return argmin_gt(gt_pl(lists, lp, ref, -1, how))


def norm_view(lists, lp, ref, min_gq, how="reference"):
    """what normcounts makes of an impure column: (state of the best genotype, second GQ >= min_gq)"""
    best, _, _ = argmin_gt(gt_pl(lists, lp, ref, -1, how))
    _, gq2, _ = argmin_gt(gt_pl(lists, lp, ref, norm_alt(lists, ref), how))
    return gt_state(GT_B1[best], GT_B2[best], ref), gq2 >= min_gq


# ---------------------------------------------------------------- columns --------------------------------------
POS = 10  # 0-based reference position of every column


def column_params(col, **over):
    args = cases.call_args(min_qv=0, min_mapq=0, qlen_lower_limit=0, qlen_upper_limit=1000, min_sequence_identity=0.0,
                           min_trim=0.0, min_bq=1, min_gq=col["min_gq"], min_ref_count=0, min_alt_count=0,
                           md_threshold=1000)
    args.update(over)
    p = gtmodel.make_params(**args)
    p.log10_prior[col["state"]] = col["lp"][col["state"]]
    return p


def column_priors(state, value):
    lp = [math.log10(v) for v in gtmodel.germline_priors(1e-3)]
    lp[state] = value
    return lp


def column_batch(col):
    """one length-1 read per entry at POS, in the column's file order (tests/test_kat.py::_site_batch)"""
    bb = pack.BatchBuilder()
    r = col["ref"]
    for i, (a, q) in enumerate(zip(col["alleles"], col["quals"])):
        cs = ":1" if a == r else "*%s%s" % (r.lower(), a.lower())
        bb.add(tstart=POS, tend=None, qstart=0, qend=None, qseq=a, bq=bytes([q]), mapq=60, is_secondary=False,
               qname="q%d" % i, cs=cs)
    return bb.finish()


def column_ref(col):
    rnd = random.Random(len(col["alleles"]) * 131 + col["quals"][0])
    s = [rnd.choice(BASES) for _ in range(64)]
    s[POS] = col["ref"]
    return "".join(s).encode()


def unpack(row):
    form, ref, alleles, quals, state, lp_hex, min_gq = row
    col = dict(form=form, ref=ref, alleles=alleles, quals=list(bytes.fromhex(quals)), state=state, min_gq=min_gq)
    col["lp"] = column_priors(state, float.fromhex(lp_hex))
    col["lists"] = allele_lists(alleles, col["quals"])
    col["r"] = BASES.index(ref)
    return col


def disagreements(col):
    """-> {mistake: (call form differs, normcounts form differs)} at the column's prior"""
    lists, lp, r, k = col["lists"], col["lp"], col["r"], col["min_gq"]
    c0, n0 = call_view(lists, lp, r), norm_view(lists, lp, r, k)
    return {m: (call_view(lists, lp, r, m) != c0, norm_view(lists, lp, r, k, m) != n0) for m in MISTAKES}


# ---------------------------------------------------------------- the search ------------------------------------
def _qualities(rnd, n, qmax):
    kind = rnd.randrange(4)
    if kind == 0:
        return [rnd.randint(1, qmax) for _ in range(n)]
    if kind == 1:
        return [93 if rnd.random() < 0.6 else rnd.randint(1, qmax) for _ in range(n)]  # the modal value and exceptions
    if kind == 2:
        return [rnd.randint(1, 25) for _ in range(n)]
    return [rnd.choice([1, 2, 7, 30, 60, 93, qmax]) for _ in range(n)]


def _random_column(rnd, form, depth, qmax):
    """a pileup with all four alleles (with two, the allele order would add x + 0.0 and y in either order: exact)"""
    r = rnd.randrange(4)
    others = [a for a in ATGC if a != r]
    rnd.shuffle(others)
    n_oth = [rnd.randint(1, max(1, depth // 6)) for _ in range(3)]
    if form == "norm":  # a clear majority alt: the allele normcounts' second GQ leaves out
        n_oth.sort(reverse=True)
        n_oth[0] = max(n_oth[0], n_oth[1] + 1)
    n_ref = max(2, depth - sum(n_oth))
    alleles = [r] * n_ref + [a for a, n in zip(others, n_oth) for _ in range(n)]
    rnd.shuffle(alleles)
    quals = _qualities(rnd, len(alleles), qmax)
    if form == "norm":  # the majority alt is the allele the second GQ skips; in the full PL it must not win
        quals = [min(q, rnd.randint(1, 12)) if a == others[0] else q for a, q in zip(alleles, quals)]
    return r, "".join(BASES[a] for a in alleles), quals


def _edge(f, lo, hi):
    """f(lo) != f(hi): bisect to adjacent doubles (lo, nextafter(lo, hi)) where f changes"""
    flo = f(lo)
    while True:
        mid = lo + (hi - lo) / 2
        if mid == lo or mid == hi:
            return lo, hi
        if f(mid) == flo:
            lo = mid
        else:
            hi = mid


def search(seed, form, count, depth=(8, 40), qmax=93):
    """knife-edge columns: -> rows (form, ref, alleles, quals hex, tuned state, its log10 prior as float hex, min_gq).

    form "call": the reference-order (best, GQ, tie) of `call` changes between the kept prior and a neighbouring
    double, and some mistake evaluator gives another result there.  form "norm": the same for normcounts' second GQ
    (alt allele skipped) against min_gq, with hom-ref the best genotype."""
    rnd = random.Random(seed)
    rows = []
    while len(rows) < count:
        r, alleles, quals = _random_column(rnd, form, rnd.randint(*depth), qmax)
        lists = allele_lists(alleles, quals)
        lp0 = column_priors(0, math.log10(gtmodel.germline_priors(1e-3)[0]))
        skip = norm_alt(lists, r) if form == "norm" else -1
        pl = gt_pl(lists, lp0, r, skip)
        best, gq, _ = argmin_gt(pl)
        if form == "norm" and gt_state(GT_B1[best], GT_B2[best], r) != HOMREF:
            continue
        second = min((g for g in range(10) if g != best), key=lambda g: pl[g])
        state = gt_state(GT_B1[second], GT_B2[second], r)
        if state == gt_state(GT_B1[best], GT_B2[best], r):
            continue  # moving that prior moves both PL
        # aim: PL[second] = PL[best] + k, k = 0 (tie / argmin edge) or an integer GQ
        k = 0 if (form == "call" and rnd.random() < 0.4) else rnd.randint(max(1, min(gq, 98) - 12), min(98, gq + 12))
        acc = -pl[second] / 10.0 - lp0[state]
        t0 = -(pl[best] + k) / 10.0 - acc
        if not -12.0 < t0 < 0.0:
            continue  # keep the prior a probability, within a few orders of magnitude of himut's
        min_gq = k if k else 20

        def view(t, how="reference"):
            lp = column_priors(state, t)
            if form == "norm":
                return norm_view(lists, lp, r, min_gq, how)
            v = call_view(lists, lp, r, how)
            return v if k else v[0::2]  # at k = 0 only the best genotype and the tie flag are the edge

        lo, hi = t0 - 1e-9 * max(1.0, abs(t0)), t0 + 1e-9 * max(1.0, abs(t0))
        if view(lo) == view(hi):
            continue
        lo, hi = _edge(view, lo, hi)
        if form == "norm" and not view(lo)[0] == view(hi)[0] == HOMREF:
            continue
        found = None
        for t in (lo, hi):
            col = dict(lists=lists, lp=column_priors(state, t), r=r, min_gq=min_gq)
            if form == "norm" and norm_view(lists, col["lp"], r, min_gq)[0] != HOMREF:
                continue
            d = disagreements(col)
            n = sum(v[0] or v[1] for v in d.values())
            if n and (found is None or n > found[0]):
                found = (n, t)
        if found:
            rows.append((form, BASES[r], alleles, bytes(quals).hex(), state, found[1].hex(), min_gq))
    return rows


# (seed, form, count, depth range, highest quality): what `search` ran to produce COLUMNS, in order.  Deep families:
# more reads than the 64 entry slots HIMUT_B200_SITE_SLOTS=64 leaves (the reduce computes the rest itself), and more
# than 255 (normcounts sends the whole span to the exact pass).  Qualities up to 250: min_bq >= 129 keeps bases.
FAMILIES = [
    (1, "call", 30, (8, 40), 93),
    (2, "norm", 16, (8, 40), 93),
    (3, "call", 3, (70, 120), 93),
    (4, "norm", 2, (70, 120), 93),
    (5, "call", 2, (256, 300), 93),
    (6, "norm", 2, (256, 300), 93),
    (7, "call", 3, (8, 40), 250),
    (8, "norm", 2, (8, 40), 250),
]


def rebuild():
    return [row for seed, form, count, depth, qmax in FAMILIES for row in search(seed, form, count, depth, qmax)]


# what rebuild() returns (python tests/test_genotype_edges.py prints it)
COLUMNS = [
    ('call', 'A', 'ACAGATACAAAAAAGT', '0101011512010d16070e18011108190f', 3, '-0x1.e03fc9743d612p+1', 34),
    ('call', 'G', 'GGGTCGGGGGGGAGGGCGGGTG', '025d5d1e1e5d02073c5d5d5d5d07011e5d3c015d023c', 1, '-0x1.70b912527da05p+1', 45),
    ('call', 'A', 'AAAGTAGAAAAAAAATTCATAAAAAATCAAAAATGACGG', '1e5d071e07013c3c3c5d3c071e3c015d025d023c3c025d015d3c5d5d5d07015d5d01015d011e01', 1, '-0x1.4af6b3b2519a4p+1', 46),
    ('call', 'T', 'TTGTCTATTT', '073c1e01073c5d1e0701', 1, '-0x1.6283e0cc8051cp-1', 20),
    ('call', 'A', 'CAAAAAAAAGAAAAGAAAAAAAGTAA', '0701025d070101015d075d3c071e1e071e0101073c1e0107025d', 1, '-0x1.9b7a66cc92601p+1', 97),
    ('call', 'G', 'GGAGCGGGGGGGTGGGGGGGGGTGTAGCGG', '20340a23470a0a035202262e403d140d412a0a42561717141329280e5b42', 1, '-0x1.d989eab3d4bc4p+1', 80),
    ('call', 'T', 'TTTCGCATTTTTTTTCTTTTTATTTT', '3c01015d073c023c0202075d071e3c1e023c01021e01023c073c', 1, '-0x1.96987428ddc72p+1', 40),
    ('call', 'T', 'TATCTTTTTGTTCATTTTTATT', '104e424a31171421371c495d074058335c522d324216', 1, '-0x1.e18e52aabb555p+0', 12),
    ('call', 'A', 'AAAAAAAAAAAGGTGACAACAAAAAAAAAAAAAA', '023c01075d3c5d5d5d5d3c021e3c5d3c1e5d5d075d021e3c5d3c02073c015d1e3c1e', 1, '-0x1.59dc28b88c2acp+1', 83),
    ('call', 'C', 'CACTCCTCCCGG', '5d5d3c07021e5d071e021e3c', 1, '-0x1.6283e0cc80518p-1', 20),
    ('call', 'G', 'ATGGGGGGC', '275445293627292e23', 1, '-0x1.630ae1aae7285p-1', 20),
    ('call', 'A', 'ACAAAAAAACTAAACAAAAAAAACAAAAATTAGGAAACCA', '183550070d4658235c0e1b2209514a44530b0a1c53174238034c303f5b251d1a4d401f373a572f46', 1, '-0x1.30ad0a2d03df5p+1', 19),
    ('call', 'T', 'TTATTTCGTTCTTTTTTTTTT', '160906101702071615030d04160f0a1611100d0414', 1, '-0x1.01a00d2c57102p+1', 67),
    ('call', 'C', 'CACCCACCCCGCCTCGC', '19040811090917080e050509070e121514', 1, '-0x1.d616d5e7b9e79p+0', 53),
    ('call', 'C', 'ACACCCCGCACCCACTCCCCCCGGCCCCCACCTC', '1c5d2b5d5d5d395d135d52025d5d115d5d3b5d5d24355d5d5d53010f5d5d475d545d', 1, '-0x1.08c052fb33d76p+2', 12),
    ('call', 'T', 'TTCTTAGTGCTTCTTTTT', '533e06431f0203283c245d36164d12485b29', 1, '-0x1.e45faafaa7cefp+1', 62),
    ('call', 'C', 'GCCTCCTCTCCCACTCGAGCCCCGGCACCCATCGCT', '5d5d023c023c1e1e5d02015d01025d5d01015d1e1e1e5d023c3c025d3c3c01025d1e0207', 1, '-0x1.24d4167b61a08p+0', 20),
    ('call', 'G', 'GGGGGATGGAGGGGGGGGGGGGGCGATGGGGCG', '015d025d1e5d3c025d5d3c075d015d015d025d3c1e5d1e3c3c0207015d025d5d3c', 1, '-0x1.80944c8719fa5p+1', 59),
    ('call', 'C', 'CCCCCTACCGTTACCCCCCTACCACCC', '191202150c1303101503120f0b111201060b0c0705130513040d0b', 3, '-0x1.ab8b7d34491e9p+1', 74),
    ('call', 'G', 'TGGGTGGGAGGGGGGGGGCGGGGGGGGGGGG', '0a5d5d5d5d5d055d5d485d5d445d1a5d5d415d5d5d5d2b4f1d525d055d065d', 1, '-0x1.f8c8b40136d60p+0', 73),
    ('call', 'A', 'ACACAAGAAAAAAAAATTA', '0110010416151316140e17130b0b03150e0717', 1, '-0x1.9b44af794160ap+1', 71),
    ('call', 'C', 'CCCCCCCCCCCGAACCCCCCCACCCCTCCACTGCTCTCAC', '0b0a13020717030b041615030519170a0e140b080115171706191919111813150c0a0a0d0e110f03', 1, '-0x1.c7af335a33841p+0', 92),
    ('call', 'A', 'GAAAAGAAATAGAAAAAAAACA', '140413150a1216090e010a1903151004110814181518', 1, '-0x1.489fb510513ffp+1', 65),
    ('call', 'T', 'CTTTTTTCGTTTTAT', '5d5d5d135d5d5d5d4d46395d5d5d5d', 1, '-0x1.4b2b6a3fa0da3p+1', 3),
    ('call', 'T', 'TTTTTTGTCGTTTTTTTTTCTATTT', '3c07021e013c075d5d3c5d073c075d3c011e071e5d0107015d', 1, '-0x1.638704d5272abp+1', 53),
    ('call', 'T', 'TCGTTTTAT', '0f38384f1c242e545d', 1, '-0x1.cbf5eb9decfd4p+1', 29),
    ('call', 'G', 'GGTGGGGAATGCGCGGGGGCGTGGGG', '011e3c5d3c5d5d1e023c3c07015d5d075d071e025d5d5d3c075d', 1, '-0x1.8edbeae696798p-1', 20),
    ('call', 'T', 'TTGTATTTTTTTTTGTCTTTTATGTATGTT', '1e3c3c07023c3c3c073c5d5d02075d025d015d07011e1e5d5d3c5d023c1e', 1, '-0x1.b42cbcc632cdbp+1', 34),
    ('call', 'G', 'GGGGGGGCGCGGGGGCGGCCGGAGGGGGGGGTGGCG', '32073c24353c2b410d163446374f3e411429132d124f191d1c3b54140e5a0e37073b1430', 1, '-0x1.428486392a53ep+1', 49),
    ('call', 'A', 'AAAAAAAACCAATAAAAAGATTAAGAAAAGCAT', '205d5d085d2d5d551b25295d56025d2d4f1d5d295d265d5d5d145d17135d5d5a5d', 1, '-0x1.1a61b6a544d7cp+1', 20),
    ('norm', 'A', 'CAACAATAAAG', '02010c040b0d0e11061206', 3, '-0x1.083e41b07a198p+1', 33),
    ('norm', 'G', 'GGGGTCGGGGAT', '085d055d035d5d5d5d5d300c', 1, '-0x1.254c04c514536p+1', 19),
    ('norm', 'C', 'TCCAGTCC', '0c3a474e06033450', 1, '-0x1.a5d305a2262c7p+1', 22),
    ('norm', 'A', 'AAAAAATAAAACAAAAGAATAA', '5d5d425b205d095d5d5021245d5d5d5d5d1f5d0b0e5d', 1, '-0x1.972db5abd1fefp+1', 58),
    ('norm', 'G', 'GGGGGCGGGGTGGGGGAGGGAAGGGGTGGGAGGGACA', '1e023c3c0101070107075d01025d1e02013c071e0201025d071e01070101013c5d070b1e02', 1, '-0x1.d139f341c74d8p+0', 81),
    ('norm', 'G', 'GCGGGGGAGGGGGCGCGGGGTGGGGGGGGGGGGGAGTAA', '040512190e040b0c0817110906060f17080d0c191318050f0f1801140d18060d110207090d090b', 1, '-0x1.69bdd24a5ed87p-1', 93),
    ('norm', 'A', 'CGCAAAGACATAATAA', '093c020701075d0707075d5d075d5d1e', 1, '-0x1.fea21de885289p+1', 11),
    ('norm', 'C', 'CTCTCACGCCCCTACCATCCC', '1e060703025d1e5d0207070201021e025d045d0702', 1, '-0x1.424b0f84192b5p+1', 15),
    ('norm', 'C', 'CCCCCACCCCACCCTCGGCCACCTTGTATCAA', '031819150e01120b08140c120a1015050c0b07100405070b09050e0c09030a01', 3, '-0x1.81228c6aec0e6p+1', 74),
    ('norm', 'A', 'AACAAATGGGACAAACAGAAAAACAAAAAAG', '01011e3c02015d0102011e071e5d5d0107015d07020201021e5d01075d5d08', 1, '-0x1.16c874fb4856dp+1', 57),
    ('norm', 'T', 'TTTGTTAGC', '11460f040e3c1c074f', 1, '-0x1.76c2567b68f45p+1', 21),
    ('norm', 'C', 'CCCCCCGACCCCCCCCCTTACTCCCCCCC', '5d5d515d5d465d1d4d5d0e5d180c3c1b5d090c5d5d073b5d5223035d5d', 1, '-0x1.c54035e96b065p+1', 70),
    ('norm', 'C', 'GCCTGCCCCCCTACCACCTC', '07120a010101070b020b120518160b0f030e0a17', 3, '-0x1.ee18f7760391ap+1', 59),
    ('norm', 'T', 'TTTGTACCTTTGTTGT', '485d120410335d255d5d5d094607055d', 1, '-0x1.02c1caf9a323ap+1', 13),
    ('norm', 'C', 'CGCCCCCCCCCCACCCCCCCCCCCACCCCCACTGCCCCCT', '5d5d5d4a5d385d535d5d2d5d0b5d5d5d395d5d5d2e05503707475d5d5d5d025d555d155d2f5d5d54', 1, '-0x1.8844e53104afcp+1', 74),
    ('norm', 'C', 'CCCCTGCCCCCCGACTTCCACGGACTCCCTCCCCGAG', '180d06180b031114100d1408060414010c010a1005030602010b0d10151401101513050807', 1, '-0x1.56c874fbbffeep+1', 93),
    ('call', 'T', 'TTTTATTTTTTTTTTTTTCTTAACTTTTTTTTTTTTTCTTTTATTTCTTTTTCTCTATTTTAATTTTGTAACTTGCACTTATTTC', '5d1e5d01013c3c5d011e5d3c073c073c0201070101013c3c01021e073c07025d015d070707025d1e1e1e5d3c1e5d5d3c5d3c013c5d3c071e5d5d5d02071e073c073c07015d1e3c07011e3c3c5d02015d5d071e075d', 1, '-0x1.d3bfbfff137d8p+1', 84),
    ('call', 'A', 'AACAAAAAAAATAAAACATAAAAGAAATCAATAACAGGCAGACAACACATTAAATAATAAACAAAAACACCAAACGTA', '5d1e5d3c1e3c5d5d0202075d02023c3c07025d5d3c5d075d5d5d1e3c5d3c3c07020701071e5d1e02023c0702071e5d5d021e5d1e5d3c021e3c5d5d5d3c011e5d015d1e5d5d011e02025d5d5d5d01', 1, '-0x1.4121b69eba369p+1', 23),
    ('call', 'T', 'TATGGTTTTTGCTTAATTTTGTGTTGTTTGTAAGTTTTTGATTGTTTACTTTTTTCTATTATTTATTTTTTGTTGTTTTTTTTTT', '0e5c1847464a332e0d2323320712063e4123205a422e2b343a46092e400f14234c0d580f490f185a1949365633114c4e13331946441649171a2130260439353229474b28524044585b27563e044d1952010e551e3f', 1, '-0x1.5c97bbd69f497p+1', 20),
    ('norm', 'A', 'AATACAAGAAAATAGAGTAAAGGCGCAAATCAGAGCGGAAAAAAATAAGCCAAAAGCAAAGCTAAGTTCAAAACTCCTAGCAACACTAAAAAATAATGAAG', '46142f4a1a403d0a0a514d1a1513025c0a4d07452d0b0a0702144617225008260a240153030144590812253606012d44052f0a1a38570b0905251a570b171a5c0b0702012643434437090c43522c5605511a425947085908091238120e432a422c0a241206', 1, '-0x1.06a7ca2435384p+2', 59),
    ('norm', 'G', 'AGGGGGGGGAGGTGGGCGGGGGAGGGGGAGCGGGGGAGGTGGGGGGACGGCGTGGGGGGGGAGAGTGGGAGGTTGTTAG', '032f0d314a1c3f2e4a06470c33150c3a32441b040c250611113b392d0329345628330e2c05420a5b3f385c301e4a09153725102b4505435157581f4f180c1e0a2e373936450b1040025a382e3d081a', 1, '-0x1.0672e6ff07127p+2', 86),
    ('call', 'G', 'GGCGGGGGGGGGGGGGGGGCCAGGGGGGAGGGTTGGGAGGGGGGGGGGGGGGGGGGTGGGCGGTGGGGTGGGGGGGGAGGGGGTGGGGGGGGGAGGGGGGTGGGAAGGGGGGGGGTGTCGGGGATGGGGTGGAGGGGGAGGGGGGGGGGAAGTGGGGTGGGATGGCGGGGGGGGGGCTGGGGGGTTGGGGGGGCGGGGGGGGGAAGAGGGGGAGAGGGGGGGGGGGGGTAAGATTGGGTGGGGTAGAAGGGGGGGTTGGGGGCGGGGGGTGAGG', '0d5d513a38105d5d5d5d5d5d155d4d5d5d585d051f5d335d5d275d5d1f5d5508345d5d5d5d5d5d251a2a5d5d5d5d5d0e5d5d5d5d5d5d5d5d5d345d4b595d5d5d5d03435d5d5d4f5d5c5d025d0a5d5d27594e1b5d5d5d5d375d5d5d5d1b4f5d5d47305d5d5d505d0a185d5d5d46365d5d5d5d5d5d2b5d5d5d5d185d5d5d2b08120a5d535d5a3e015d5d5d5d0e5d5d5d1847510e5d1a5d5d5d0b5d3c5d5d5d5d405d5d3f5d035d5d5d2c5d5d5d0c5d5d5d435d5d230a5d475d46205d5d01135d5d5d5d5d5d5d5d395d5d4d585d5d5d415d5d534c5d5d3538315d16135d5d0a1c5d5d5d5d5d160a5d5d145d5d295d5d5d505d5d5d5d305d5d5d5a5d5d5d5d5d475d1f125d5d125d085d365d1f081f5d5d5d5d5d', 1, '-0x1.3d8afffd485e0p+1', 96),
    ('call', 'G', 'CGGGGGGGGGGGGGCGGGGGGGGGGCGGGGGGGGGCGGGTGGGATCGGCGCGCGCGGGGGGGTAGAGGTGGGGGGGAGGGGGGGTCGGAGGGGGGGCGGGGGGCGCGGGGGGGGGGGGGGGGGGCGCTGGGGGGGGTGGGGGGCGATGCGGGGGGGGGGGGGGTCGGGAGAGGTGGTGGGGGGGGGTCGGCGCGAGGGGGAGGGGGGGGGGGGGCGGGGGGGGGAGATGGGGGGGGCCGAGAGGGAGGGGGGGCGTGGGGGACTCGGGGGCGGGGGGGGGGCGGGGGGGGA', '1259075d395d5d195d5d5d5d5d4a4d215d5d525d3b5d5d5d2c5d5d465d5c5d5d5d5d5d09315d5d225d1b165d4b5d5d5d5d5d365d5d285d5d205d5d5d415d5d1f0f5d5d5d5d5d305d341d5d5d06114d5d015d5d5d5d354b5d1b5d5d5d39575d145d4e392c5d165d5d5d5d5d535d5d5d5d5d5d155d5d5d3d5d285d5d51124b5d481c5d5d5d5d5d175d5d5a5d0e5d5d5d5d595d5d5d5d5d355d5d095d395d365d5d5d12205d5d56135d465d5d2f545d5d5d105d5d5d5d265d5d5d5d5d595d5d1f18255d5d3f5d5d105d335d5d5d5d165d23345d5d5d5d5d5d325d015d5d5d5a4d145d1e3b51255d5d085d5d5d5d465d5c4e5d4c5d5d095d5d5d5d5d2e5d155d1a5d5d5a5d5d5d5d025d5d3a5d5d5d5d5d5d5d5d135d5d5d195a5d3e5d5d415d5d5d5d5d5d', 1, '-0x1.52b61fae53d80p-1', 91),
    ('norm', 'A', 'ACAATCCGCCTTAAAAAAAACACAAAAACAATAAAAAAAATTAAAAAAAACAAACTAAAAAAACATGTAACTCAAAAAACTAAGAAAATTACAACAAACTAAAAAAAAAAAAAAATCAAAACAAAACAAAAAAATTAAAAAAAAAATCATCAAAAACCAAAACTAAAACACAAAAAAAAAACAAATAACACAAAAGAAACAAAATACCAGGCAAAAAACAAAAATAAAAGAAACAAGAACAACCAAACCAAATAAAAATAACAACAAATCAAATAAA', '5d015d5d5d0c0a5d05063a2a44335d3d0d415d1b0a350c375d5d3a5d0b5d5d17425d5d5d5d5d5d493e5d2e5d5d5d2c5d5d1c095d5d5d0a2e531446415d5a5d035d5d4b5d5d49035d0c5d5d5d363b5d0c5d5d5d225d5d4c5d5d4757015d14045d585d0a5d423e5d5d54564d035d2e5d5d5d185d480b5d043137025d5d5d1705185d5d4a5d5d2e5d5b5d5d4d3c5d5d5d5d53535d04242907035d5c5d5d0407025d5d5d075d4c5d5d5d095d0a5d0b035d5d115d5d5d5d0c5d055d01445d051605325d055d5d5d5d1a095d5b5d545d5d030b442b420a5d5d5d5d292f075d5d2b125d5d411b5d5d5d5d5b5d02505d5d5d05045820040930340c02074b5d5d39215a285d5d053c39085d02085d5d5d5d015d5d5d5d5d2e32', 1, '-0x1.973817f173910p+1', 63),
    ('norm', 'T', 'TTAATTATTAATTTGCTTTAGTATTCTTTTTTTTTTGTGTTTTTGTTTTCTTTTTTTTTTTCTTTGTTTTTTTTTTGTTTCGTTTTTTTTTGTTTTGTTTTTTTATTGTTTATGGGTTTTTTTTATTTTTTTTTTTTTTTTTTTTTTTTTTTTTGTTTTTTCTTTTTTATCTATTTTGATTTTATTGCTTTTTTTTTTTTGTTAGATTTTGCTGTCTGTCTTTTGATTTCTTATTTTCTTTGGTTATGATTTTTATGGTTTTTTTTTTTTTTATTTTTTTTTATTT', '435d5d395d015d555c5d5d5d5d5d032f2e5d1d5d013a585d105d225d175d5d365d5d505d0a3f0a57515d0415075d5d10215d5d5d5d5d48015d5d0b5d5d5d5d5d5d074c5d575d5d5d5d0f1c5d0c325d5d1c025d5d5d5d5d5d5d485d023d5d5d5d06235d5d5d5c58445d5d0e024b5d5d515d0a07085d5d1b5d2d5d4a355d38335d5d5d4e5d1c5d5d2803485d5d5d5d5d5d5d5d5d2f5d5d5d535d52043c495d5d5d125d5d5d15502e5d5d3f5d5d5d1b3f5d010a5d5d285d5d235d5d0a1e5d4c1f5d3d575d5d5d4e4f5d03445d5d085d5d5d5d1e015d5d02540f5d03355d485d5d5d065d5d5d5d0e5c5d5d41445d5d5d20145d06065d5d5d15095d5d5d3b3a5d5d5801045d165d5d5d5d5d5d5d49475d5d5d5d5d2c5c5d3a4c435d5d5d5d5d5d', 1, '-0x1.12f713beae470p+1', 83),
    ('call', 'T', 'TTTTGTTATTTTTTGCTTTTTTTGTTTT', '5d5d5d1b5d605d915d5d6e785d5d5db3155d5dbb5d135d5d276c5dc4', 1, '-0x1.630e40dbc399cp+1', 13),
    ('call', 'A', 'AAAAAAAAAAGAATATCAAAAGCCAG', '0192278a1af35e9e0713e0369e6127a341f5599b5e7a201eda7d', 0, '-0x1.f232341214681p-4', 65),
    ('call', 'C', 'TCCCCTCTACCCCCCCCCCCCCCGCCCCCTTCCTCGCC', '1801010910090717140c0f180c0c0308040810070b071014140110150c150316040d17190710', 3, '-0x1.a77969f806b93p+1', 80),
    ('norm', 'G', 'GATGGGGGGGCCGGCGGGGGGG', '1e1e5d015d0701fa011e09041e010a0107025d011e5d', 1, '-0x1.174f75e6aa8cap+1', 45),
    ('norm', 'A', 'TTACAGAACACA', '3c3c020702073c070c5d01fa', 1, '-0x1.3f075750b6118p+1', 9),
]

CHUNK = [(0, 64)]


def columns():
    return [unpack(row) for row in COLUMNS]


def flip(best, ref):
    """the genotype a record shows: ref allele first (gtlib.py:133-134)"""
    g0, g1 = GT_B1[best], GT_B2[best]
    return (g1, g0) if g0 != ref and ((g0 == ref) + (g1 == ref)) == 1 else (g0, g1)


def norm_counter(col):
    """the normcounts log counter the column's reads land in (normcounts.py:317-400): 3 / 4 / 5 het / hetalt / homalt,
    10 GQ below min_gq, 13 counted"""
    state, gq_ok = norm_view(col["lists"], col["lp"], col["r"], col["min_gq"])
    return {HET: 3, HETALT: 4, HOMALT: 5}.get(state, 13 if gq_ok else 10)


def test_restatement_matches_the_oracle():
    """pins the restatement (and which reads' qualities enter the lists) to the oracle on every column, both forms"""
    for i, col in enumerate(columns()):
        p, b = column_params(col), column_batch(col)
        chunks = b.chunk_table(CHUNK)
        rec, _ = oracle.call_chunks(p, b, chunks)
        best, gq, tie = call_view(col["lists"], col["lp"], col["r"])
        assert rec.size == sum(1 for a in ATGC if a != col["r"] and col["lists"][a]), i
        for x in rec:
            assert int(x["gq"]) == gq, i
            assert bool(x["flags"] & abi.SITE_PL_TIE) == tie, i
            assert tuple(int(v) for v in x["germ_gt"]) == flip(best, col["r"]), i
            assert int(x["germ_state"]) == gt_state(GT_B1[best], GT_B2[best], col["r"]), i
        _, _, log, _ = oracle.normcounts_chunks(p, b, column_ref(col), chunks)
        n, c = len(col["alleles"]), norm_counter(col)
        assert int(log[1]) == n and int(log[c]) == n, (i, list(log))


def test_every_column_sits_on_an_edge():
    """the stored prior is one double away from another reference-order result"""
    for i, col in enumerate(columns()):
        view = (lambda lp: norm_view(col["lists"], lp, col["r"], col["min_gq"])) if col["form"] == "norm" else \
            (lambda lp: call_view(col["lists"], lp, col["r"]))
        t = col["lp"][col["state"]]
        here = view(col["lp"])
        assert any(view(column_priors(col["state"], math.nextafter(t, d))) != here for d in (-math.inf, math.inf)), i


def test_the_edge_set_is_not_vacuous():
    cols = columns()
    assert len(cols) >= 40
    for m in MISTAKES:
        d = [disagreements(col)[m] for col in cols]
        assert sum(c for c, _ in d) >= 3, (m, "call form")
        assert sum(n for _, n in d) >= 3, (m, "normcounts form")
    # the three kinds of boundary in `call`: GQ at an integer, a tie flag that flips, another best genotype
    kinds = set()
    for col in cols:
        ref = call_view(col["lists"], col["lp"], col["r"])
        for m in MISTAKES:
            alt = call_view(col["lists"], col["lp"], col["r"], m)
            kinds.add("argmin" if alt[0] != ref[0] else "tie" if alt[2] != ref[2] else "gq" if alt[1] != ref[1] else None)
    assert {"argmin", "tie", "gq"} <= kinds
    for form in ("call", "norm"):
        depths = [len(c["alleles"]) for c in cols if c["form"] == form]
        assert max(depths) > 255 and any(64 < n <= 255 for n in depths), form
    assert any(max(c["quals"]) > 128 for c in cols)


# ---------------------------------------------------------------- the certificate, restated ---------------------
CERT_PRIORS = (1e-3, 1e-2, 5e-4, 0.3)


def homref_with_gq(quals, prior, min_gq):
    """a pure column of these qualities, file order: hom-ref and GQ >= min_gq in the reference's arithmetic?"""
    lp = [math.log10(v) for v in gtmodel.germline_priors(prior)]
    best, gq, _ = call_view((list(quals), [], [], []), lp, 0)
    return best == 0 and gq >= min_gq


@pytest.mark.parametrize("min_bq", [1, 20, 60, 93])
def test_certified_pure_columns_at_the_threshold(min_bq):
    """k_norm_bits certifies depth n once the callable count reaches thr[n]; the quality sum it assumes is the least
    one: callable bases at exactly min_bq, the others at 1 and at min_bq - 1.  Every such column at thr[n] - 1,
    thr[n], thr[n] + 1 that passes must be hom-ref with GQ >= min_gq."""
    n_cert = n_not = 0
    for prior in CERT_PRIORS:
        for min_gq in (0, 20, 60, 99):
            cert = test_norm_cert.make_cert(prior, min_gq, min_bq)
            assert cert is not None
            thr = cert["thr"]
            assert thr[:cert["n_min"]] == [0xffff] * cert["n_min"]
            assert all(a <= b for a, b in zip(thr[cert["n_min"]:], thr[cert["n_min"] + 1:]))
            for n in range(1, 256):
                for cal in {thr[n] - 1, thr[n], thr[n] + 1} if thr[n] <= n else {n}:
                    if not 0 <= cal <= n:
                        continue
                    if cal < thr[n]:
                        n_not += 1
                        continue
                    assert test_norm_cert.certified_sum(cert, n, min_bq * cal + (n - cal)), (prior, min_gq, n, cal)
                    for fill in {1, max(min_bq - 1, 1)}:
                        n_cert += 1
                        quals = (min_bq,) * cal + (fill,) * (n - cal)
                        assert homref_with_gq(quals, prior, min_gq), (prior, min_gq, min_bq, n, cal, fill)
    if min_bq > 1:  # at min_bq 1 the bound is s1 >= n whatever cal is: almost no thr[n] exists
        assert n_cert > 1000 and n_not > 1000


@pytest.mark.parametrize("prior", CERT_PRIORS)
def test_certified_random_pure_columns(prior):
    """the 30 000 random pure positions of test_norm_cert.py (same seeds, same draws), held against the restatement
    instead of the reference's own gtlib (which is not part of the repository)"""
    for min_gq in (0, 5, 20, 60, 99):
        cert = test_norm_cert.make_cert(prior, min_gq)
        rnd = random.Random(hash((prior, min_gq)) & 0xffff)
        n_cert = n_not = 0
        for _ in range(1500):
            n = rnd.choice([1, 2, 3, 5, 8, 13, 20, 30, 45, 80, 150, 255]) if rnd.random() < 0.5 else rnd.randrange(1, 256)
            bqs = test_norm_cert.quality_mix(rnd, n)
            rnd.choice("ATGC")  # that test's reference base: the model is symmetric in it, the draw keeps the stream
            if not test_norm_cert.certified(cert, bqs):
                n_not += 1
                continue
            n_cert += 1
            assert homref_with_gq(tuple(bqs), prior, min_gq), (n, bqs[:8], min_gq)
        assert n_not > 0
        if min_gq < 99 and prior < 0.1:
            assert n_cert > 200


# ---------------------------------------------------------------- every route on the GPU ------------------------
def same_norm(g, o):
    return np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1]) and list(g[2]) == list(o[2]) and g[3] == o[3]


def kernels(ctx):
    return [n for n, _ in ctx.last_kernel_times()]


@pytest.mark.gpu
def test_call_routes_match_the_oracle(ctx, monkeypatch):
    from himut_b200 import bamdec
    for i, col in enumerate(columns()):
        p, b = column_params(col), column_batch(col)
        chunks = b.chunk_table(CHUNK)
        o_rec, o_log = oracle.call_chunks(p, b, chunks)
        ctx.set_params(p)
        ctx.set_site_sets()
        got = {}
        ctx.upload(b)
        got["fused"] = ctx.call_chunks(chunks)
        assert ctx.last_call_path() == 2, i
        monkeypatch.setenv("HIMUT_B200_CALL_V1", "1")  # the route of chunks of 2^27 positions and more
        got["v1"] = ctx.call_chunks(chunks)
        assert ctx.last_call_path() == 1, i
        monkeypatch.delenv("HIMUT_B200_CALL_V1")
        ctx.upload(b.without_seq())
        got["without_seq"] = ctx.call_chunks(chunks)
        got["compact"] = ctx.call_batch_compact(b, bamdec.compact_bq(b), chunks)
        monkeypatch.setenv("HIMUT_B200_SITE_SLOTS", "64")  # read at upload: deeper columns leave slots to the reduce
        ctx.upload(b)
        got["slots_64"] = ctx.call_chunks(chunks)
        assert ctx.last_call_path() == 2, i
        monkeypatch.delenv("HIMUT_B200_SITE_SLOTS")
        for route, (rec, log) in got.items():
            ok, why = parity.records_equal(rec, o_rec)
            assert ok, (i, route, why)
            assert list(log) == list(o_log), (i, route)


NORM_ROUTES = [  # (environment, kernels that must have run)
    ({}, ("k_norm_bits", "k_norm_entries_bits")),
]


@pytest.mark.gpu
def test_normcounts_production_routes_match_the_oracle(ctx, monkeypatch):
    from himut_b200 import bamdec
    for i, col in enumerate(columns()):
        p, b, ref = column_params(col), column_batch(col), column_ref(col)
        chunks = b.chunk_table(CHUNK)
        o = oracle.normcounts_chunks(p, b, ref, chunks)
        ctx.set_params(p)
        ctx.set_site_sets()
        ctx.upload(b)
        for env, names in NORM_ROUTES:
            for k, v in env.items():
                monkeypatch.setenv(k, v)
            g = ctx.normcounts_chunks(ref, chunks)
            ran = kernels(ctx)
            for k in env:
                monkeypatch.delenv(k)
            assert same_norm(g, o), (i, env, g, o)
            assert all(n in ran for n in names), (i, env, ran)
        # bitmap of the modal quality + exceptions: the exact pass gathers "modal wherever the bitmap says so"
        ctx.upload_compact(b, bamdec.compact_bq(b))
        g = ctx.normcounts_chunks(ref, chunks)
        assert same_norm(g, o), (i, "compact", g, o)
        assert "k_norm_entries_bits" in kernels(ctx), i
        monkeypatch.setenv("HIMUT_B200_SITE_SLOTS", "64")
        ctx.upload(b)
        g = ctx.normcounts_chunks(ref, chunks)
        monkeypatch.delenv("HIMUT_B200_SITE_SLOTS")
        assert same_norm(g, o), (i, "slots_64", g, o)


@pytest.mark.gpu
@pytest.mark.parametrize("min_bq", [0, 129])
def test_normcounts_outside_the_certified_domain(ctx, min_bq):
    """make_norm_cert turns the certificate off (min_bq 0, or above 128 with qualities up there in some columns):
    production runs the single-pass k_norm_tiles_tma"""
    for i, col in enumerate(columns()):
        p, b, ref = column_params(col, min_bq=min_bq), column_batch(col), column_ref(col)
        chunks = b.chunk_table(CHUNK)
        ctx.set_params(p)
        ctx.set_site_sets()
        ctx.upload(b)
        g = ctx.normcounts_chunks(ref, chunks)
        assert "k_norm_tiles_tma" in kernels(ctx), i
        o = oracle.normcounts_chunks(p, b, ref, chunks)
        assert same_norm(g, o), (i, g, o)


# ---------------------------------------------------------------- pure columns at the certificate's edge (GPU) --
def pure_edge_batch(cert, min_bq, depths):
    """one window of columns per depth n, each in a 1024-position span of its own: n reads span the window, and
    column by column the first `cal` reads carry min_bq, the others `fill` (1 or min_bq - 1), for cal at thr[n] - 1,
    thr[n], thr[n] + 1.  Every second window also has three short reads that touch its 32-position word but not its
    columns, so that the kernel looks thr up at a depth above the column's (k_norm_bits certifies a pure column of
    depth n and callable count c when n >= n_min and c >= thr[reads touching its word]).
    -> (batch, reference, certified window columns, window columns for the exact pass, windows with short reads)"""
    rnd = random.Random(min_bq * 1000 + len(depths))
    ref = "".join(rnd.choice(BASES) for _ in range(1024 * (len(depths) + 1)))
    bb = pack.BatchBuilder()
    thr = cert["thr"]
    n_yes = n_no = n_touched = 0
    for k, n in enumerate(depths):
        base = 1024 * k + 16
        cals = sorted({c for c in (thr[n] - 1, thr[n], thr[n] + 1) if 0 <= c <= n} if thr[n] <= n else {n - 1, n})
        cols = [(c, f) for c in cals for f in sorted({1, max(min_bq - 1, 1)})]
        touch = 3 if k % 2 and n + 3 <= 255 else 0  # more than 255 reads in a span: all of it goes to the exact pass
        n_touched += touch > 0
        for j in range(touch):
            bb.add(tstart=base - 14, tend=None, qstart=0, qend=None, qseq=ref[base - 14:base - 12], bq=bytes([93, 93]),
                   mapq=60, is_secondary=False, qname="t%d_%d" % (k, j), cs=":2")
        for j in range(n):
            bq = bytes(min_bq if j < c else f for c, f in cols)
            bb.add(tstart=base, tend=None, qstart=0, qend=None, qseq=ref[base:base + len(cols)], bq=bq, mapq=60,
                   is_secondary=False, qname="r%d_%d" % (k, j), cs=":%d" % len(cols))
        for c, _ in cols:
            if c > 0:
                if n >= cert["n_min"] and c >= thr[min(n + touch, 255)]:
                    n_yes += 1
                else:
                    n_no += 1
    return bb.finish(), ref.encode(), n_yes, n_no, n_touched


@pytest.mark.gpu
@pytest.mark.parametrize("prior,min_gq,min_bq", [(1e-3, 20, 20), (1e-3, 60, 60), (5e-4, 99, 93), (1e-2, 0, 30)])
def test_pure_columns_at_the_certificate_edge(ctx, prior, min_gq, min_bq):
    cert = test_norm_cert.make_cert(prior, min_gq, min_bq)
    depths = sorted({max(cert["n_min"], 1), cert["n_min"] + 1, 2, 5, 17, 40, 100, 200, 255})
    b, ref, n_yes, n_no, n_touched = pure_edge_batch(cert, min_bq, depths)
    assert n_yes > 0 and n_no > 0
    p = gtmodel.make_params(**cases.call_args(min_qv=0, min_mapq=0, qlen_lower_limit=0, qlen_upper_limit=1000,
                                              min_sequence_identity=0.0, min_trim=0.0, md_threshold=1000,
                                              germline_snv_prior=prior, min_gq=min_gq, min_bq=min_bq))
    chunks = b.chunk_table([(0, len(ref))])
    ctx.set_params(p)
    ctx.set_site_sets()
    ctx.upload(b)
    g = ctx.normcounts_chunks(ref, chunks)
    assert "k_norm_bits" in kernels(ctx)
    o = oracle.normcounts_chunks(p, b, ref, chunks)
    assert same_norm(g, o), (g, o)
    # the near-edge columns split: those below the threshold went to the exact pass, the others did not.  Nothing else
    # can go there but the two positions of the short reads of a window (depth 3: certified or not)
    exact = ctx.last_norm_exact_sites()
    assert n_no <= exact <= n_no + 2 * n_touched, (exact, n_no, n_yes, n_touched)


if __name__ == "__main__":  # prints COLUMNS
    print("COLUMNS = [")
    for row in rebuild():
        print("    %r," % (row,))
    print("]")
