"""The fused `himut call` path (csrc/callfused.cuh) on both sides of each of its fixed capacities, at the exact value,
and at chromosome-scale coordinates.

Each capacity picks one of two routes:
  HC_MAX_OPS = 96         k_call_scan stages a read's ops or reads the op_t / op_q prefixes k_call_pairs wrote;
  HM_BYREAD_MAX_OPS = 192 the same bound of the first version;
  HC_SITES = 64           a pair's register site list, then the 32-lane direct loop;
  HC_A_CAP = 6144         a k_call_pairs CTA stages the op words of its active pairs, or walks global memory;
  HC_TILE = 2^17          sort tile rel >> 17, (span >> 17) + 1 tiles per chunk;
  HC_CAPD = 4096          (ref, alt) masks of a tile in shared memory or in the chunk's global scratch;
  HC_STAGE = 8192         a tile's non-hole keys staged, or re-walked from the segment;
  HC_KEY_POS_BITS = 27    chunk span < 2^27 takes the fused path, wider spans the first version;
  site cap                the distinct sites fit the buffers, or the call runs again with larger ones.
Batches are built by hand (cs strings through pack.BatchBuilder) so that each case sits exactly at its edge.  Each
test checks on the host that it reached the edge, and compares records (every field) and all 15 counters with the
CPU oracle.  Most cases run on four routes: with the base stream, without it, a compact upload the call is
submitted behind, and the forced first version.  GPU."""
import numpy as np
import pytest

import cases
import parity
from himut_b200 import abi, bamdec, gtmodel, pack, synth
from oracle import oracle

pytestmark = pytest.mark.gpu

HC_MAX_OPS, HM_BYREAD_MAX_OPS, HC_SITES, HC_A_CAP = 96, 192, 64, 6144
HC_TILE, HC_CAPD, HC_STAGE, HC_KEY_POS_BITS = 1 << 17, 4096, 8192, 27
CHR1 = 248_956_422  # GRCh38 chr1

# every designed substitution becomes a candidate: no read-level or window gate
RELAXED = dict(gtmodel.DEFAULT_CALL_ARGS, qlen_lower_limit=0, qlen_upper_limit=10**9, min_trim=0,
               max_mismatch_count=10**5, min_sequence_identity=0)
P_RELAXED = gtmodel.make_params(**RELAXED)
P_DEFAULT = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
ROUTES = ("seq", "noseq", "compact", "v1")


# ---------------------------------------------------------------------------------------------------- batch helper
def random_ref(n, seed):
    rng = np.random.default_rng(seed)
    return np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n, dtype=np.uint8)].tobytes().decode()


def other_base(b, k=0):
    """the (k % 3)-th base that differs from b"""
    alts = [x for x in "ACGT" if x != b]
    return alts[k % 3]


def _tokens(start, end, ev):
    """ev: {pos: "S<alt>" | "D"} plus {("I", pos)}: insertion before pos -> cs tokens (one per op)"""
    ins = sorted(p for p in ev if isinstance(p, tuple))
    occ = sorted(p for p in ev if not isinstance(p, tuple))
    marks = sorted([(p[1], 0, p) for p in ins] + [(p, 1, p) for p in occ])
    out, cur = [], start
    for pos, _o, key in marks:
        if pos > cur:
            out.append(("M", cur, pos - cur))
            cur = pos
        if isinstance(key, tuple):
            out.append(("I", pos, 1))
        else:
            out.append((ev[key][0], pos, ev[key][1:]))
            cur = pos + 1
    if cur < end:
        out.append(("M", cur, end - cur))
    return out


def _fill_ops(start, end, ev, n_ops):
    """add 1-base deletions (+2 ops each, in the middle of the longest match run) and, for an odd gap, an insertion
    right after one of them (+1) until the read has exactly n_ops ops"""
    gap = n_ops - len(_tokens(start, end, ev))
    if gap < 0:
        raise ValueError("%d ops designed, %d asked" % (n_ops + -gap, n_ops))
    if gap == 1:  # an insertion in front of a substitution that follows a match run
        subs = [p for p in ev if not isinstance(p, tuple) and p > start and (p - 1) not in ev and ("I", p) not in ev]
        if not subs:
            raise ValueError("no place for a single insertion")
        ev[("I", subs[-1])] = None
        return
    odd = gap % 2 == 1
    while gap >= 2:
        runs = [t for t in _tokens(start, end, ev) if t[0] == "M"]
        m = max(runs, key=lambda t: t[2])
        if m[2] < 3 + (1 if odd else 0):
            raise ValueError("no match run left to split")
        p = m[1] + m[2] // 2
        ev[p] = "D"
        gap -= 2
        if odd:
            ev[("I", p + 1)] = None
            gap -= 1
            odd = False


def hand_batch(ref, reads, seed=0):
    """reads: dicts with start, length, subs [(pos, alt)] (0-based reference positions), optional n_ops (exact op
    count), end_ins (one inserted base after the last aligned one), secondary, qname.
    -> (abi.ReadBatch, one {pos: alt} per read in file order: the substitutions it carries)"""
    rng = np.random.default_rng(seed)
    bb = pack.BatchBuilder()
    carried = []
    for i, rd in sorted(enumerate(reads), key=lambda x: (x[1]["start"], x[0])):
        start, end = rd["start"], rd["start"] + rd["length"]
        ev = {}
        for pos, alt in rd.get("subs", ()):
            assert start <= pos < end and alt != ref[pos], (i, pos)
            ev[pos] = "S" + alt
        if rd.get("n_ops") is not None:
            _fill_ops(start, end, ev, rd["n_ops"])
        if rd.get("end_ins"):  # an insertion after the read's last base: it lands at rpos = tend
            ev[("I", end)] = None
        cs, qseq = [], []
        for kind, pos, val in _tokens(start, end, ev):
            if kind == "M":
                cs.append(":%d" % val)
                qseq.append(ref[pos:pos + val])
            elif kind == "S":
                cs.append("*%s%s" % (ref[pos].lower(), val.lower()))
                qseq.append(val)
            elif kind == "D":
                cs.append("-" + ref[pos].lower())
            else:
                cs.append("+c")
                qseq.append("C")
        q = "".join(qseq)
        bq = np.where(rng.random(len(q)) < 0.85, 93, rng.integers(5, 93, len(q))).astype(np.uint8)
        bb.add(tstart=start, tend=end, qstart=0, qend=len(q), qseq=q, bq=bq.tobytes(), mapq=60,
               is_secondary=bool(rd.get("secondary")), qname=rd.get("qname", "h%d" % i), cs="".join(cs))
        carried.append({p: ev[p][1:] for p in ev if not isinstance(p, tuple) and ev[p][0] == "S"})
        if rd.get("n_ops") is not None:
            assert len(_tokens(start, end, ev)) == rd["n_ops"]
    return bb.finish(), carried


def _fetched(batch, chunk):
    s, e = int(chunk[0]), int(chunk[1])
    return [r for r in range(batch.n_reads)
            if not batch.flags[r] & abi.READ_SECONDARY and batch.tstart[r] < e and batch.tend[r] > s]


def designed_keys(batch, carried, ref, chunk):
    """the site keys (tpos, ref code, alt code) of the substitutions that the non-secondary reads fetched by the chunk
    carry inside it: what k_site_sort makes distinct and k_call_scan lists per pair"""
    s, e = int(chunk[0]), int(chunk[1])
    return {(p + 1, abi.BASE2CODE[ref[p]], abi.BASE2CODE[a])
            for r in _fetched(batch, chunk) for p, a in carried[r].items() if s <= p + 1 <= e}


def key_slots(batch, carried, chunk):
    """candidate keys before they are made distinct: one per (read, substitution) inside the chunk"""
    s, e = int(chunk[0]), int(chunk[1])
    return sum(1 for r in _fetched(batch, chunk) for p in carried[r] if s <= p + 1 <= e)


def site_keys(rec):
    return set(zip(rec["tpos"].tolist(), rec["ref"].tolist(), rec["alt"].tolist()))


# ---------------------------------------------------------------------------------------------------- routes
def _oracle(p, batch, chunks):
    o_rec, o_log = oracle.call_chunks(p, batch, chunks)
    return o_rec, list(o_log)


def _same(rec, log, want, what):
    ok, why = parity.records_equal(rec, want[0])
    assert ok, "%s: %s" % (what, why)
    assert list(log) == want[1], what


def run_route(ctx, route, p, batch, chunks, monkeypatch):
    """one call of `batch` over `chunks` on the given route -> (records, log, path)"""
    ctx.set_params(p)
    ctx.set_site_sets()
    if route == "seq":
        rec, log = ctx.call_batch(batch, chunks)
    elif route == "noseq":
        rec, log = ctx.call_batch(batch.without_seq(), chunks)
    elif route == "compact":  # upload_compact not waited for, the call submitted straight behind it
        b = batch.without_seq()
        cq = bamdec.compact_bq(b)
        ctx.upload_compact(b, cq, wait=False)
        ctx.call_chunks_submit(chunks)
        rec, log = ctx.call_chunks_collect(view=False)
        ctx.upload_wait()
    else:
        monkeypatch.setenv("HIMUT_B200_CALL_V1", "1")
        try:
            rec, log = ctx.call_batch(batch, chunks)
        finally:
            monkeypatch.delenv("HIMUT_B200_CALL_V1")
    return rec, log, ctx.last_call_path()


def all_routes(ctx, p, batch, chunks, monkeypatch, routes=ROUTES, fused=True):
    """every route against the oracle; fused: the unforced routes take the fused path (else the first version)"""
    want = _oracle(p, batch, chunks)
    for route in routes:
        rec, log, path = run_route(ctx, route, p, batch, chunks, monkeypatch)
        assert path == (1 if route == "v1" or not fused else 2), route
        _same(rec, log, want, route)
    return want[0], want[1]


def check_sites(rec, batch, carried, ref, chunks):
    """the designed site keys are exactly the records' keys (relaxed gates, chunks that do not overlap)"""
    want = set()
    for ch in chunks:
        want |= designed_keys(batch, carried, ref, (ch["start"], ch["end"]))
    assert want and site_keys(rec) == want


# ---------------------------------------------------------------------------------------------------- ops per read
def _spread(start, end, k):
    """k positions from start to end - 1, both ends included, as evenly as integers allow"""
    if k == 1:
        return [start]
    return [start + (end - 1 - start) * j // (k - 1) for j in range(k)]


OPS_PATTERN = [96, 97, 95, 128, 97, 96, 191, 192, 193, 96, 97, 95, 128, 96, 97, 193, 192, 191, 95, 96, 97, 128, 96, 97]


@pytest.fixture(scope="module")
def ops_case():
    """12 kb reads every 500 bp; each has substitutions at its first and last reference position, and exactly the
    op count of OPS_PATTERN (reads 0 - 3, one k_call_scan CTA of four warps, hold a 96- and a 97-op read); the
    designed substitutions are >= 21 bp apart, so the default gates hold them too"""
    n = 30_000
    ref = random_ref(n, 1)
    reads = []
    for i, k in enumerate(OPS_PATTERN):
        start, length = 1000 + 500 * i, 12_000 + 7 * i
        n_sub = (k + 1) // 2 if k % 2 else k // 2 - 1  # odd: subs and runs alternate; even: + deletion + insertion
        subs = [(p, other_base(ref[p], p)) for p in _spread(start, start + length, n_sub)]
        reads.append(dict(start=start, length=length, subs=subs, n_ops=k))
    batch, carried = hand_batch(ref, reads, seed=1)
    return batch, carried, ref, n


def test_ops_per_read_at_the_staging_bounds(ctx, ops_case, monkeypatch):
    batch, carried, ref, n = ops_case
    ops = batch.n_ops.tolist()
    assert {95, 96, 97, 128, 191, 192, 193} <= set(ops)
    assert {HC_MAX_OPS, HC_MAX_OPS + 1} <= set(ops[:4]) and {HM_BYREAD_MAX_OPS - 1, HM_BYREAD_MAX_OPS, HM_BYREAD_MAX_OPS + 1} <= set(ops)
    chunks = batch.chunk_table([(0, n)])
    assert chunks["read_lo"][0] == 0  # pair index == read index: reads 0 - 3 are one k_call_scan CTA
    for r in range(batch.n_reads):  # candidate sites at both ends of every op list
        ts, te = int(batch.tstart[r]), int(batch.tend[r])
        assert ts in carried[r] and te - 1 in carried[r]
    rec, _ = all_routes(ctx, P_RELAXED, batch, chunks, monkeypatch)
    check_sites(rec, batch, carried, ref, chunks)
    rec, log = all_routes(ctx, P_DEFAULT, batch, chunks, monkeypatch)
    assert rec.size > 500 and log[0] == batch.n_reads


# ---------------------------------------------------------------------------------------------------- sites per pair
SITES_PER_PROBE = [1, 31, 32, 33, 63, 64, 65, 95, 96, 97, 129]


@pytest.fixture(scope="module")
def sites_case():
    """one region per count K: a 12 kb probe read without substitutions whose range [ts + 1, te + 1] holds exactly K
    site keys (K > 1: the last at rpos = te, where the probe has no base, only the insertion it ends with), two 16 kb
    carrier reads that make them (the same alt inside the probe's range), a plain read; sites at tpos = ts and te + 2,
    just outside the probe's range, with two alts each"""
    step = 22_000
    n = 5_000 + step * len(SITES_PER_PROBE) + 5_000
    ref = random_ref(n, 2)
    reads, probes = [], []
    for j, k in enumerate(SITES_PER_PROBE):
        ts = 5_000 + step * j + 3_000
        te = ts + 12_000
        inside = _spread(ts, te - 600, k) if k == 1 else _spread(ts, te - 600, k - 1) + [te]
        pos = sorted(set(inside) | {ts - 1, te + 1})
        probes.append((ts, te, k))
        reads.append(dict(start=ts - 2_000, length=16_000, subs=[(p, other_base(ref[p], 0)) for p in pos]))
        reads.append(dict(start=ts - 1_500, length=15_000,
                          subs=[(p, other_base(ref[p], 0 if ts <= p <= te else 1)) for p in pos]))
        reads.append(dict(start=ts - 1_000, length=14_000))
        reads.append(dict(start=ts, length=te - ts, end_ins=True, qname="probe%d" % k))
    batch, carried = hand_batch(ref, reads, seed=2)
    return batch, carried, ref, n, probes


def test_sites_per_pair_around_the_register_list(ctx, sites_case, monkeypatch):
    batch, carried, ref, n, probes = sites_case
    chunks = batch.chunk_table([(0, n)])
    keys = designed_keys(batch, carried, ref, (0, n))
    in_range = lambda ks, ts, te: [k for k in ks if ts + 1 <= k[0] <= te + 1]  # what k_call_scan lists for the probe
    for ts, te, k in probes:
        r = int(np.flatnonzero((batch.tstart == ts) & (batch.tend == te))[0])
        assert not carried[r]
        assert len(in_range(keys, ts, te)) == k
        assert k == 1 or any(t == te + 1 for t, _, _ in keys)
        assert sum(t == ts for t, _, _ in keys) == 2 and sum(t == te + 2 for t, _, _ in keys) == 2  # just outside
    assert {k for _, _, k in probes} >= {HC_SITES - 1, HC_SITES, HC_SITES + 1, HC_SITES + 33}
    rec, _ = all_routes(ctx, P_RELAXED, batch, chunks, monkeypatch)
    check_sites(rec, batch, carried, ref, chunks)
    got = site_keys(rec)
    for ts, te, k in probes:
        assert len(in_range(got, ts, te)) == k
    all_routes(ctx, P_DEFAULT, batch, chunks, monkeypatch)


# ---------------------------------------------------------------------------------------------------- CTA op span
def _ops_read(ref, start, length, n_ops, **kw):
    n_sub = (n_ops + 1) // 2 if n_ops % 2 else n_ops // 2 - 1
    subs = [(p, other_base(ref[p], p)) for p in _spread(start, start + length, n_sub)]
    return dict(start=start, length=length, subs=subs, n_ops=n_ops, **kw)


@pytest.fixture(scope="module")
def span_case():
    """batch A: three k_call_pairs CTAs (128 pairs each) whose reads hold 6143, 6144 and 6145 op words.
    batch B: one CTA whose first pair is a secondary read and whose last pair a read that ends before the chunk
    (both with long op lists); the 126 active pairs between them hold exactly 6144 op words"""
    n = 16_000
    ref = random_ref(n, 3)
    per_cta = [[48] * 127 + [47], [48] * 128, [48] * 127 + [49]]
    reads = [_ops_read(ref, 100 + 20 * i, 1_500, k) for i, k in enumerate(sum(per_cta, []))]
    a, ca = hand_batch(ref, reads, seed=3)
    reads = [_ops_read(ref, 0, 12_000, 301, secondary=True)]
    reads += [_ops_read(ref, 100 + 10 * i, 4_000, 49 if i <= 96 else 48) for i in range(1, 127)]
    reads.append(_ops_read(ref, 100 + 127 * 10, 600, 199))
    b, cb = hand_batch(ref, reads, seed=4)
    return ref, (a, ca, n), (b, cb)


def test_cta_op_span_at_the_stage_bound(ctx, span_case, monkeypatch):
    ref, (a, ca, n), _ = span_case
    chunks = a.chunk_table([(0, n)])
    assert chunks["read_lo"][0] == 0 and chunks["read_hi"][0] == 3 * 128
    spans = [int(a.op_off[128 * k + 127] + a.n_ops[128 * k + 127] - a.op_off[128 * k]) for k in range(3)]
    assert spans == [HC_A_CAP - 1, HC_A_CAP, HC_A_CAP + 1]
    rec, _ = all_routes(ctx, P_RELAXED, a, chunks, monkeypatch)
    check_sites(rec, a, ca, ref, chunks)


def test_cta_op_span_from_active_pairs_only(ctx, span_case, monkeypatch):
    ref, _, (b, cb) = span_case
    chunks = b.chunk_table([(2_000, 12_000)])
    assert b.n_reads == 128 and chunks["read_lo"][0] == 0 and chunks["read_hi"][0] == 128
    assert b.flags[0] & abi.READ_SECONDARY and b.tend[127] <= 2_000  # the CTA's first and last pairs are inactive
    assert all(b.tend[r] > 2_000 and not b.flags[r] & abi.READ_SECONDARY for r in range(1, 127))
    assert int(b.op_off[126] + b.n_ops[126] - b.op_off[1]) == HC_A_CAP
    assert int(b.op_off[127] + b.n_ops[127] - b.op_off[0]) > HC_A_CAP
    rec, _ = all_routes(ctx, P_RELAXED, b, chunks, monkeypatch)
    check_sites(rec, b, cb, ref, chunks)


# ---------------------------------------------------------------------------------------------------- sort tiles
@pytest.mark.parametrize("span", [HC_TILE - 1, HC_TILE, HC_TILE + 1])
def test_sort_tile_boundaries(ctx, span, monkeypatch):
    """sites at rel = -1, 0, 2^17 - 1, 2^17, 2^17 + 1, span and span + 1 of one chunk; with span = 2^17 the second
    tile holds rel = 2^17 alone"""
    S = 20_000
    n = S + span + 20_000
    ref = random_ref(n, 5)
    rels = sorted({-1, 0, HC_TILE - 1, HC_TILE, HC_TILE + 1, span, span + 1})
    designed = [S + r - 1 for r in rels]  # tpos = S + rel
    reads = []
    for centre in (S, S + HC_TILE):
        for i in range(6):
            start = centre - 6_500 + 1_000 * i
            subs = [(p, other_base(ref[p], i)) for p in designed if start <= p < start + 12_000 and i % 2 == 0]
            subs += [(p, other_base(ref[p], 1)) for p in range(start + 150 + 37 * i, start + 12_000, 400)
                     if all(abs(p - d) > 30 for d in designed)]
            reads.append(dict(start=start, length=12_000, subs=subs))
    batch, carried = hand_batch(ref, reads, seed=5)
    chunks = batch.chunk_table([(S, S + span)])
    got = {t for t, _, _ in designed_keys(batch, carried, ref, (S, S + span))}
    in_chunk = sorted(t - S for t in got if t - S in rels)
    assert in_chunk == [r for r in rels if 0 <= r <= span]
    n_tiles = (span >> 17) + 1
    if span == HC_TILE:
        assert n_tiles == 2 and [t - S for t in got if (t - S) >> 17 == 1] == [HC_TILE]
    rec, _ = all_routes(ctx, P_RELAXED, batch, chunks, monkeypatch)
    check_sites(rec, batch, carried, ref, chunks)
    all_routes(ctx, P_DEFAULT, batch, chunks, monkeypatch)


# ---------------------------------------------------------------------------------------------------- tile capacities
def _region_reads(ref, a, region, positions, alt_of, every, length=5_000, step=1_000):
    """reads of `length` every `step` bp over [a, a + region); every: each read covering a position carries it, else
    only the last read that starts at or before it"""
    reads = []
    for s in range(a, a + region - length + 1, step):
        subs = [(p, alt_of(p)) for p in positions if s <= p < s + length and (every or p - s < step)]
        reads.append(dict(start=s, length=length, subs=subs))
    return reads


@pytest.mark.parametrize("every", [True, False], ids=["keys_unstaged", "keys_staged"])
def test_distinct_positions_per_tile(ctx, every, monkeypatch):
    """three chunks of one tile each, with 4095, 4096 and 4097 distinct candidate positions (the (ref, alt) masks
    fit in shared memory, fit exactly, spill to the chunk's global scratch); each position carried by every read that
    covers it (about 20 000 keys per tile: more than the stage holds), or by one read (the tile's keys staged)"""
    counts = [HC_CAPD - 1, HC_CAPD, HC_CAPD + 1]
    region, gap = 70_000, 100_000
    n = gap * len(counts) + 10_000
    ref = random_ref(n, 6)
    reads, loci = [], []
    for j, d in enumerate(counts):
        a = 10_000 + gap * j
        positions = [a + 5_000 + 12 * i for i in range(d)]
        reads += _region_reads(ref, a, region, positions, lambda p: other_base(ref[p], p // 12), every)
        loci.append((a, a + region))
    batch, carried = hand_batch(ref, reads, seed=6)
    chunks = batch.chunk_table(loci)
    for (s, e), d in zip(loci, counts):
        got = designed_keys(batch, carried, ref, (s, e))
        assert len(got) == d and max(got)[0] - s < HC_TILE  # one tile
        slots = key_slots(batch, carried, (s, e))
        assert slots > HC_STAGE if every else slots == d
    rec, _ = all_routes(ctx, P_RELAXED, batch, chunks, monkeypatch)
    check_sites(rec, batch, carried, ref, chunks)


P_HOLES = gtmodel.make_params(**dict(RELAXED, max_mismatch_count=1, mismatch_window=2))


def test_keys_per_tile(ctx, monkeypatch):
    """three one-tile chunks with 8191, 8192 and 8193 candidate keys that pass (duplicates: up to three reads per
    position, two alts), and clusters of three adjacent substitutions that fail the mismatch-window test (their
    slots are holes, which the stage does not count)"""
    targets = [HC_STAGE - 1, HC_STAGE, HC_STAGE + 1]
    length, step, spacing = 3_000, 500, 20
    gap = 120_000
    n = gap * len(targets) + 10_000
    ref = random_ref(n, 7)
    rng = np.random.default_rng(7)
    reads, loci, want_keys = [], [], []
    for j, target in enumerate(targets):
        a = 10_000 + gap * j
        m = (target + 2) // 3
        positions = [a + length + spacing * i for i in range(m)]  # six reads cover every position
        region = positions[-1] - a + length
        starts = list(range(a, a + region - length + 1, step))
        subs = {s: [] for s in starts}
        keys = 0
        for i, p in enumerate(positions):
            k = 3 if i < m - 1 else target - 3 * (m - 1)
            cover = [s for s in starts if s <= p < s + length]
            for c, s in enumerate(cover[:k]):
                subs[s].append((p, other_base(ref[p], c % 2)))
            keys += min(k, len(cover))
        for s in starts:  # holes: three adjacent substitutions in the middle of gaps the read covers whole
            for p in positions:
                h = p + 9
                if s <= h and h + 2 < s + length and rng.random() < 0.15:
                    subs[s] += [(h + u, other_base(ref[h + u], u)) for u in range(3)]
        reads += [dict(start=s, length=length, subs=subs[s]) for s in starts]
        loci.append((a, a + region))
        want_keys.append(keys)
    assert want_keys == targets
    batch, carried = hand_batch(ref, reads, seed=7)
    chunks = batch.chunk_table(loci)
    for (s, e), target in zip(loci, targets):
        assert e - s < HC_TILE
        fetched = [r for r in range(batch.n_reads) if batch.tstart[r] < e and batch.tend[r] > s]
        isolated = holes = 0
        for r in fetched:
            pos = sorted(carried[r])
            for i, p in enumerate(pos):
                near = (i > 0 and p - pos[i - 1] <= 4) or (i + 1 < len(pos) and pos[i + 1] - p <= 4)
                holes += near
                isolated += not near
        assert isolated == target and holes > 1_000
    rec, _ = all_routes(ctx, P_HOLES, batch, chunks, monkeypatch)
    want = set()
    for r in range(batch.n_reads):
        pos = sorted(carried[r])
        for i, p in enumerate(pos):
            if not ((i > 0 and p - pos[i - 1] <= 4) or (i + 1 < len(pos) and pos[i + 1] - p <= 4)):
                want.add((p + 1, abi.BASE2CODE[ref[p]], abi.BASE2CODE[carried[r][p]]))
    assert site_keys(rec) == want


# ---------------------------------------------------------------------------------------------------- site cap
@pytest.mark.parametrize("delta", [-1, 0, 1])
def test_site_cap_retry_at_its_exact_value(ctx, delta, monkeypatch):
    d = synth.generate(60_000, seed=41)
    chunks = d.batch.chunk_table([(0, 60_000)])
    want = _oracle(P_DEFAULT, d.batch, chunks)
    n_sites = want[1][1]
    assert n_sites == want[0].size > 100
    ctx.set_params(P_DEFAULT)
    ctx.set_site_sets()
    ctx.upload(d.batch)
    monkeypatch.setenv("HIMUT_B200_SITE_CAP", str(n_sites + 1))
    rec, log = ctx.call_chunks(chunks)
    one_pass = ctx.last_timing()[1]
    _same(rec, log, want, "cap n + 1")
    monkeypatch.setenv("HIMUT_B200_SITE_CAP", str(n_sites + delta))
    rec, log = ctx.call_chunks(chunks)
    assert ctx.last_call_path() == 2
    _same(rec, log, want, "cap n %+d" % delta)
    assert ctx.last_timing()[1] == (2 * one_pass if delta < 0 else one_pass)  # the overflow ran the call twice


# ---------------------------------------------------------------------------------------------------- shifted batches
def shifted(batch, off):
    """the same reads `off` positions further along the contig (ops are relative to tstart)"""
    kw = {name: getattr(batch, name) for name, _ in abi.ReadBatch._FIELDS}
    assert int(batch.tend.max()) + off < 2**31
    kw["tstart"] = (batch.tstart.astype(np.int64) + off).astype(np.int32)
    kw["tend"] = (batch.tend.astype(np.int64) + off).astype(np.int32)
    return abi.ReadBatch(**kw)


@pytest.fixture(scope="module")
def synth60():
    return synth.generate(60_000, seed=43)


def test_span_route_at_2_27_without_forcing(ctx, synth60, monkeypatch):
    off = 2**27 - 40_000
    b = shifted(synth60.batch, off)
    assert b.tstart.min() < 2**27 < b.tend.max()
    cases_ = [((0, 2**27 - 1), 2), ((0, 2**27), 1), ((2**27 - 50_000, 2**27 + 50_000), 2)]
    for (s, e), path in cases_:
        assert (e - s >= 1 << HC_KEY_POS_BITS) == (path == 1)
        chunks = b.chunk_table([(s, e)])
        rec, _ = all_routes(ctx, P_DEFAULT, b, chunks, monkeypatch, routes=("seq", "noseq"), fused=path == 2)
        assert rec.size > 50
        if e == 2**27 - 1:  # rel = tpos - 0 near the top of the 32-bit relative key
            assert rec["tpos"].max() > 2**27 - 20_000


def test_span_route_at_2_28(ctx, synth60, monkeypatch):
    off = 2**28 - 30_000
    b = shifted(synth60.batch, off)
    assert b.tstart.min() < 2**28 < b.tend.max()
    chunks = b.chunk_table([(0, 2**28 + 5)])  # first version, 29 position bits in its keys
    rec, _ = all_routes(ctx, P_DEFAULT, b, chunks, monkeypatch, routes=("seq", "noseq"), fused=False)
    assert b.tend[: chunks["read_hi"][0]].max() > 2**28  # fetched reads reach past 2^28
    assert rec.size > 50 and rec["tpos"].max() > 2**28 - 1_000


# ---------------------------------------------------------------------------------------------------- many chunks
def _mixed_loci(rng, k, n):
    """k windows over a contig of n: empty (past the contig), negative spans, one-position and zero-length windows,
    the rest overlapping windows of up to 3 kb"""
    out = []
    for i in range(k):
        kind = int(rng.integers(0, 8))
        p = int(rng.integers(1, n - 1))
        if kind == 0:
            out.append((n + 1_000 + p, n + 1_500 + p))
        elif kind == 1:
            out.append((p, p - int(rng.integers(1, 3_000))))
        elif kind == 2:
            out.append((p, p + 1))
        elif kind == 3:
            out.append((p, p))
        else:
            out.append((p, min(n, p + int(rng.integers(2, 3_000)))))
    return out


@pytest.mark.parametrize("k", [1, 7, 8, 9, 63, 64, 65, 511, 512, 513, 4100])
def test_many_chunks(ctx, k, monkeypatch):
    n = 100_000
    d = synth.generate(n, seed=44, depth=10.0)
    loci = _mixed_loci(np.random.default_rng(k), k, n)
    if k == 1:
        loci = [(0, n)]
    chunks = d.batch.chunk_table(loci)
    assert len(chunks) == k
    if k >= 63:  # every kind is there
        empty = chunks["read_lo"] == chunks["read_hi"]
        span = chunks["end"].astype(np.int64) - chunks["start"]
        assert empty.any() and (span < 0).any() and (span == 1).any() and (span == 0).any()  # empty: pair_off repeats
    rec, log = all_routes(ctx, P_DEFAULT, d.batch, chunks, monkeypatch, routes=("seq", "v1"))
    assert log[0] > 0


def test_reads_per_chunk_around_powers_of_8(ctx, monkeypatch):
    """chunks (0, e) whose read ranges hold 1, 7, 8, 9, 63, 64, 65, 511, 512 and 513 reads: the searches of
    k_site_range2 over the chunk's reads at and around the depths of the 8-ary search"""
    n = 100_000
    d = synth.generate(n, seed=45, depth=100.0)
    ts, nr = d.batch.tstart, d.batch.n_reads
    pmax = np.maximum.accumulate(d.batch.tend)
    want = [1, 7, 8, 9, 63, 64, 65, 511, 512, 513]
    for j in range(nr):  # a start past the reads that share tstart = 0: the chunk's first read is read lo
        s = int(pmax[j])
        lo = int(np.searchsorted(pmax, s, side="right"))
        if all(lo + k < nr and ts[lo + k - 1] < ts[lo + k] for k in want):
            break
    loci = [(s, int(ts[lo + k])) for k in want]
    chunks = d.batch.chunk_table(loci)
    assert (chunks["read_hi"] - chunks["read_lo"]).tolist() == want
    all_routes(ctx, P_DEFAULT, d.batch, chunks, monkeypatch, routes=("seq", "noseq", "v1"))


# ---------------------------------------------------------------------------------------------------- chromosome scale
N_CHROM = 300_000
OFFSETS = [2**26 + 12_345, 2**27 - 100_000, CHR1 - N_CHROM, 2**28 - 50_000]


@pytest.fixture(scope="module")
def chrom():
    """the unshifted contig, its chunks and calls, and a random ACGT prefix long enough for every offset"""
    d = synth.generate(N_CHROM, seed=46)
    loci = cases.chunkloci(0, N_CHROM)
    assert len(loci) == 2
    chunks = d.batch.chunk_table(loci)
    rec, log = oracle.call_chunks(P_DEFAULT, d.batch, chunks)
    codes = np.random.default_rng(46).integers(0, 4, max(OFFSETS), dtype=np.uint8)
    prefix = np.frombuffer(b"ACGT", np.uint8)[codes].tobytes()
    return d, loci, parity.sort_records(rec), list(log), prefix


def _shift_loci(loci, off):
    return [(s + off, e + off) for s, e in loci]


def _translated(rec, base, off):
    """rec equals base with tpos + off and every other field identical"""
    rec, moved = parity.sort_records(rec), base.copy()
    moved["tpos"] += off
    ok, why = parity.records_equal(rec, moved)
    assert ok, why


@pytest.mark.parametrize("off", OFFSETS)
def test_call_at_chromosome_scale(ctx, chrom, off, monkeypatch):
    d, loci, base_rec, base_log, _ = chrom
    b = shifted(d.batch, off)
    assert int(b.tstart.max()) > off and int(b.tstart.min()) >= off
    chunks = b.chunk_table(_shift_loci(loci, off))
    assert (chunks["read_lo"] == d.batch.chunk_table(loci)["read_lo"]).all()
    rec, log = all_routes(ctx, P_DEFAULT, b, chunks, monkeypatch)
    _translated(rec, base_rec, off)
    assert log == base_log and rec.size > 100


@pytest.mark.parametrize("off", OFFSETS)
def test_normcounts_at_chromosome_scale(ctx, chrom, off):
    """the reference is `off` random bases followed by the contig, so the packed reference and the trinucleotide
    table of the bit-vector pass cover the whole length; chunks that avoid the contig's first and last base count
    what they count unshifted"""
    d, loci, _, _, prefix = chrom
    p = P_DEFAULT
    ref = prefix[:off] + d.ref
    b = shifted(d.batch, off)
    inner = [(1_000, 150_000), (150_000, N_CHROM - 1_000)]
    ctx.set_params(p)
    ctx.set_site_sets()
    ctx.upload(d.batch)
    base = ctx.normcounts_chunks(d.ref, d.batch.chunk_table(inner))
    for lo in (_shift_loci(loci, off), _shift_loci(inner, off)):
        chunks = b.chunk_table(lo)
        ctx.upload(b)
        g = ctx.normcounts_chunks(ref, chunks)
        assert "k_norm_bits" in [k for k, _ in ctx.last_kernel_times()]
        o = oracle.normcounts_chunks(p, b, ref, chunks)
        assert np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1]) and list(g[2]) == list(o[2]) and g[3] == o[3]
    assert np.array_equal(g[0], base[0]) and np.array_equal(g[1], base[1]) and list(g[2]) == list(base[2]) and g[3] == base[3]
    assert int(g[0].sum()) > 0


@pytest.mark.parametrize("off", OFFSETS)
def test_device_bam_decode_at_chromosome_scale(ctx, chrom, off, tmp_path):
    """BAI bins above level 1 and a linear index of up to ~15 000 windows: the device decode equals the host decode
    and the batch; `call` on it and normcounts on the decode with bases match the oracle"""
    d, loci, base_rec, base_log, prefix = chrom
    b = shifted(d.batch, off)
    path = str(tmp_path / "s.bam")
    bamdec.write_batch_bam(path, "chr1", off + N_CHROM + 1_000, b)
    nb = bamdec.NativeBam(path, threads=2)
    try:
        s, e = off, off + N_CHROM
        host = nb.read_batch("chr1", s, e, seq=True)
        want = nb.read_batch("chr1", s, e, seq=False)
        region = ctx.decode_region(nb, "chr1", s, e)
        got = ctx.read_back()
        assert region.n_reads == b.n_reads == got.n_reads
        for name in ("tstart", "tend", "qstart", "qlen", "mapq", "qname_id", "bq_off", "op_off", "n_ops", "bq", "ops"):
            x, y = getattr(got, name), getattr(want, name)
            assert x.shape == y.shape and np.array_equal(x, y), name
        for name in ("tstart", "tend", "qstart", "qlen", "mapq", "bq_off", "op_off", "n_ops", "bq", "ops"):
            assert np.array_equal(getattr(got, name), getattr(b, name)), name
        chunks = region.chunk_table(_shift_loci(loci, off))
        ctx.set_params(P_DEFAULT)
        ctx.set_site_sets()
        rec, log = ctx.call_chunks(chunks)
        assert ctx.last_call_path() == 2
        _same(rec, log, _oracle(P_DEFAULT, host, chunks), "device decode")
        _translated(rec, base_rec, off)
        ctx.decode_region(nb, "chr1", s, e, seq=True)
    finally:
        nb.close()
    ref = prefix[:off] + d.ref
    g = ctx.normcounts_chunks(ref, chunks)
    assert "k_norm_bits" in [k for k, _ in ctx.last_kernel_times()]
    o = oracle.normcounts_chunks(P_DEFAULT, host, ref, chunks)
    assert np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1]) and list(g[2]) == list(o[2]) and g[3] == o[3]
