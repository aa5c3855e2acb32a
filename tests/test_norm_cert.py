"""The certified verdict of the normcounts integer pass (DESIGN.md §4.1) against the reference's own genotype code:
whenever the integer test (restated here from make_norm_cert in himut_b200.cu, which turns it into the table thr that
k_norm_bits looks up) certifies a pure position — n reads of the reference allele with qualities b_i — the unmodified
`himut.gtlib.get_germ_gt` must call it hom-ref with GQ >= min_gq.  Random depths, quality mixes, priors and GQ
thresholds.  The comparisons with the reference run where its unmodified sources are present (tests/refshim.py)."""
import math
import random

import pytest

import refshim
from himut_b200 import gtmodel

needs_reference = pytest.mark.skipif(not refshim.have_reference(), reason="reference sources are not present")


def make_cert(prior, min_gq, min_bq=93):
    """make_norm_cert (himut_b200/csrc/himut_b200.cu) restated -> dict or None (bit-vector pass switched off)"""
    p = gtmodel.make_params(**dict(gtmodel.DEFAULT_CALL_ARGS, germline_snv_prior=prior, min_gq=min_gq, min_bq=min_bq))
    L2 = 0.30102999566398119521
    f1 = -p.lut_hom[1]
    if not (1 <= min_bq <= 128 and min_gq <= 99 and 0.0 < f1 < 1.0):
        return None
    for bq in range(1, 256):
        hom, het, err = p.lut_hom[bq], p.lut_het[bq], p.lut_err[bq]
        if not (hom <= 0.0) or not (abs(het - (hom - L2)) <= 1e-9) or not (abs(err + bq / 30.0) <= 1e-9):
            return None
        if not (-hom <= f1 * (255 - bq) / 254.0 + 1e-12):
            return None
    margin = 1e-6
    need = (float(min_gq) if min_gq > 0 else 0.0) + margin
    lp = list(p.log10_prior)
    c_het = 10.0 * (lp[0] - lp[1])
    n_min = max(1.0, math.ceil((need + margin - c_het) / (10.0 * L2)))
    if n_min > 1e6:
        return None
    a_bq = 10.0 / 30.0 * (1.0 - 1e-12)
    a_x = 10.0 * f1 / 254.0 * (1.0 + 1e-12)
    c_oth = 10.0 * (lp[0] - max(lp[2], lp[3])) - margin
    cert = dict(n_min=int(n_min), ia_bq=math.floor(a_bq * 1048576.0), ia_x=math.ceil(a_x * 1048576.0),
                i_need=math.ceil((need - c_oth) * 1048576.0))
    # thr[n]: the smallest callable count that certifies depth n from the lower bound s1 >= min_bq cal + (n - cal)
    # (k_norm_bits), made non-decreasing in n; 0xffff: none
    thr, run = [], 0
    for n in range(256):
        t = 0xffff
        if n >= cert["n_min"]:
            t = next((cal for cal in range(n + 1) if certified_sum(cert, n, min_bq * cal + (n - cal))), 0xffff)
            t = run = max(t, run)
        thr.append(t)
    cert["thr"] = thr
    return cert


def certified_sum(cert, n, s1):
    """the integer test on depth n and quality sum s1 (without the depth bound n >= n_min)"""
    x = min(254 * n, 255 * n - s1)
    return s1 * cert["ia_bq"] - x * cert["ia_x"] >= cert["i_need"]


def certified(cert, bqs):
    """the fixed-point test of make_norm_cert (himut_b200.cu: `n >= c.n_min`, `s1 * c.ia_bq - x * c.ia_x >= c.i_need`)"""
    return len(bqs) >= cert["n_min"] and certified_sum(cert, len(bqs), sum(bqs))


def quality_mix(rnd, n):
    kind = rnd.randrange(6)
    if kind == 0:
        return [93] * n
    if kind == 1:
        return [93 if rnd.random() < 0.9 else rnd.randrange(1, 94) for _ in range(n)]
    if kind == 2:
        return [rnd.randrange(1, 94) for _ in range(n)]
    if kind == 3:
        return [rnd.randrange(1, 12) for _ in range(n)]          # poor reads only
    if kind == 4:
        return [rnd.choice([1, 2, 93]) for _ in range(n)]          # extremes of the convexity bound
    return [rnd.randrange(1, 256) for _ in range(n)]               # beyond what PacBio writes


@needs_reference
@pytest.mark.parametrize("prior", [1e-3, 1e-2, 5e-4, 0.3])
@pytest.mark.parametrize("min_gq", [0, 5, 20, 60, 99])
def test_certified_positions_are_homref_with_enough_gq(prior, min_gq):
    himut = refshim.import_reference()
    himut.gtlib.np = refshim.StableArgsortNumpy()
    himut.gtlib.init(prior)
    cert = make_cert(prior, min_gq)
    assert cert is not None
    rnd = random.Random(hash((prior, min_gq)) & 0xffff)
    n_cert = n_not = 0
    for _ in range(1500):
        n = rnd.choice([1, 2, 3, 5, 8, 13, 20, 30, 45, 80, 150, 255]) if rnd.random() < 0.5 else rnd.randrange(1, 256)
        bqs = quality_mix(rnd, n)
        ref = rnd.choice("ATGC")
        if not certified(cert, bqs):
            n_not += 1
            continue
        n_cert += 1
        lists = {0: [], 1: [], 2: [], 3: [], 4: [], 5: []}
        lists[himut.util.base2idx[ref]] = bqs
        gt, gq, state, _ = himut.gtlib.get_germ_gt(ref, lists)
        assert state == "homref" and gt == ref + ref, (n, bqs[:8], gt, state)
        assert gq >= min_gq, (n, sum(bqs), gq, min_gq)
    assert n_not > 0
    if min_gq < 99 and prior < 0.1:
        assert n_cert > 200  # the test is not vacuous: typical pileups are certified


def test_thirty_reads_at_q93_are_certified_by_default():
    assert certified(make_cert(1e-3, 20), [93] * 30)
    assert certified(make_cert(1e-3, 20), [93])            # the prior alone puts het 30 above hom-ref
    assert not certified(make_cert(1e-3, 60), [93] * 5)    # 5 reads: 15 + 30 < 60
    assert make_cert(1e-3, 20, min_bq=200) is None           # outside the certified domain: exact pass only


@needs_reference
def test_every_table_entry_is_the_references_value():
    """the per-BQ terms and priors the kernels add are the reference's own functions' values, bit for bit, over the whole
    table (tests/test_kat.py pins four entries without the reference)"""
    himut = refshim.import_reference()
    hom, het, err = gtmodel.bq_tables()
    for bq in range(1, 256):
        assert hom[bq] == himut.gtlib.get_log10_one_minus_epsilon(bq)
        assert het[bq] == himut.gtlib.get_log10_one_half_minus_epsilon(bq)
        assert err[bq] == himut.gtlib.get_log10_epsilon(bq / 3)
    for prior in (1e-3, 1e-2, 5e-4, 0.3, 0.00123):
        himut.gtlib.init(prior)
        ours = gtmodel.germline_priors(prior)
        for state, v in zip(("homref", "het", "hetalt", "homalt"), ours):
            assert math.log10(v) == himut.gtlib.get_log10_germ_gt_prior(state), (prior, state)
