"""The three DEFLATE decoders of the BAM readers on streams zlib's encoder never writes (deflate_enc.py builds them,
zlib.decompress proves each one valid): the host decoder of inflate_fast.h alone (hm_inflate_raw, no zlib fallback)
and two streams at a time (hm_inflate_raw2), and the device decoder of k_bgzf_inflate (inflate_block, through
k_inflate_one).  Each stream is at most 65 536 bytes out, the BGZF limit."""
import collections
import os
import random
import re
import zlib

import pytest

import deflate_enc as de
import test_inflate as ti


def _rnd_bytes(rnd, n, alphabet=None):
    return bytes(rnd.choice(alphabet) for _ in range(n)) if alphabet else rnd.randbytes(n)


def _tail():
    """short matches and literals at the very end: the host decoder leaves its fast path there (16 input bytes, 320
    output bytes left)"""
    return [(3, 1), 65, (4, 2), (5, 7), 66, (6, 16), (10, 33), (3, 300), (7, 5), 67, (3, 3), (8, 9), (4, 1), (3, 17)] * 3


def _fixed_lengths():
    rnd = random.Random(1)
    toks = list(_rnd_bytes(rnd, 300))
    for k in range(29):
        lo = de.LEN_BASE[k]
        hi = min(lo + (1 << de.LEN_EXTRA[k]) - 1, 257)  # 258 is code 285
        toks += [(lo, 1 + k), rnd.randrange(256), (hi, 200 + k), rnd.randrange(256)]
    return [{"type": "fixed", "tokens": toks + _tail()}]


def _fixed_distances():
    rnd = random.Random(2)
    toks = list(_rnd_bytes(rnd, 33_000))
    for k in range(30):
        lo = de.DIST_BASE[k]
        hi = lo + (1 << de.DIST_EXTRA[k]) - 1
        toks += [(3, lo), rnd.randrange(256), (4, hi), rnd.randrange(256)]
    toks += [(258, 32768), (3, 32768)]
    return [{"type": "fixed", "tokens": toks + _tail()}]


def _fixed_overlaps():
    rnd = random.Random(3)
    toks = list(_rnd_bytes(rnd, 20))
    for d in range(1, 18):
        for n in (3, 15, 16, 17, 258):
            toks += [(n, d), rnd.randrange(256)]
    return [{"type": "fixed", "tokens": toks + _tail()}]


def _stored_empty_everywhere():
    rnd = random.Random(4)
    a = _rnd_bytes(rnd, 3000, b"ACGT")
    b = _rnd_bytes(rnd, 3000, b"ACGTN")
    return [{"type": "stored", "data": b""}, {"type": "fixed", "tokens": de.tokenize(a)}, {"type": "stored", "data": b""},
            {"type": "dynamic", "tokens": de.tokenize(a + b, len(a))}, {"type": "stored", "data": b""}]


def _stored_full():
    rnd = random.Random(5)
    return [{"type": "stored", "data": _rnd_bytes(rnd, 65535)}, {"type": "stored", "data": b"\x7f"}]


def _stored_after_fixed(pad):
    rnd = random.Random(6)
    a = _rnd_bytes(rnd, 2000, b"ACGT!#")
    toks = de.tokenize(a)
    while (_bits_of_fixed(toks) + 3) % 8 == 0:  # a 9-bit literal until the stored block's header leaves bits to pad
        toks.append(200)
    return [{"type": "fixed", "tokens": toks}, {"type": "stored", "data": _rnd_bytes(rnd, 700), "pad": pad},
            {"type": "fixed", "tokens": [(5, 700), 66] + _tail()}]


def _bits_of_fixed(toks):
    n = 3 + 7  # header + end of block
    for t in toks:
        if isinstance(t, int):
            n += de.FIXED_LIT[t]
        else:
            s, eb, _ = de.len_symbol(t[0])
            _, deb, _ = de.dist_symbol(t[1])
            n += de.FIXED_LIT[s] + eb + 5 + deb
    return n


def _dyn_literal_only_257():
    rnd = random.Random(7)
    data = _rnd_bytes(rnd, 20_000, bytes(range(200)))
    return [{"type": "dynamic", "tokens": list(data)}]


def _dyn_286_30_crossing18():
    """matches only at distances >= 1025 and of lengths 3-10: the literal/length lengths end in zeros and the distance
    lengths begin with them, one 18 run across the boundary"""
    rnd = random.Random(8)
    base = _rnd_bytes(rnd, 2000)
    toks = list(base)
    out = bytearray(base)
    while len(out) < 60_000:
        if rnd.random() < 0.3:
            n, d = rnd.randrange(3, 11), rnd.randrange(1025, min(len(out), 32768) + 1)
            toks.append((n, d))
            for _ in range(n):
                out.append(out[-d])
        else:
            b = rnd.randrange(256)
            toks.append(b)
            out.append(b)
    return [{"type": "dynamic", "tokens": toks + [(3, 1025)], "hlit": 286, "hdist": 30, "combined": True}]


def _dyn_crossing16():
    """one run of 9-bit lengths from the last literal/length symbol into the first six distance symbols: a 16 run
    across the boundary; literal/length and distance codes of 9 bits"""
    lit = [8] * 226 + [9] * 60
    dist = [9] * 6 + [1, 2, 3, 4, 5, 6, 9, 9] + [0] * 16
    rnd = random.Random(9)
    data = _rnd_bytes(rnd, 300, bytes(range(226)))
    data += b"".join(data[rnd.randrange(0, 250):][:rnd.randrange(3, 40)] + bytes([rnd.randrange(226)]) for _ in range(1500))
    toks = de.tokenize(data, window=128)
    return [{"type": "dynamic", "tokens": toks + [(258, 1), (3, 6)], "lit_lens": lit, "dist_lens": dist, "hlit": 286, "hdist": 30,
             "combined": True}]


def _dyn_long_codes():
    """literal/length and distance codes of 1-15 bits (a chain: one code of each length, two of 15), every code used;
    the distance codes of 9-15 bits are the host decoder's distance subtables"""
    rnd = random.Random(10)
    lits = list(range(65, 75))
    lsyms = lits[:5] + [256] + lits[5:] + [257, 258, 259, 260, 261]
    lit_lens = de.chain_lengths(lsyms, 286)
    dist_lens = de.chain_lengths(list(range(16)), 30)
    toks = [rnd.choice(lits) for _ in range(400)]
    out = bytearray(toks)
    plan = [("l", s) for s in lits] + [("m", s) for s in (257, 258, 259, 260, 261)] + [("d", k) for k in range(16)]
    plan += [("l", rnd.choice(lits)) for _ in range(600)] + [("d", rnd.randrange(16)) for _ in range(200)]
    rnd.shuffle(plan)
    for kind, s in plan:
        if kind == "l":
            toks.append(s)
            out.append(s)
            continue
        n = (3 + (s - 257)) if kind == "m" else rnd.randrange(3, 8)
        k = rnd.randrange(16) if kind == "m" else s
        d = rnd.randrange(de.DIST_BASE[k], de.DIST_BASE[k] + (1 << de.DIST_EXTRA[k]))
        toks.append((n, d))
        for _ in range(n):
            out.append(out[-d])
    return [{"type": "dynamic", "tokens": toks + [(3, 1)] + [65] * 3, "lit_lens": lit_lens, "dist_lens": dist_lens}]


def _dyn_precode7_hclen19():
    """a code-length code with 7-bit codes, all 19 of its lengths sent"""
    rnd = random.Random(11)
    data = bytes(min(255, int(rnd.expovariate(0.02))) for _ in range(30_000))
    return [{"type": "dynamic", "tokens": de.tokenize(data), "skew": True, "hclen": 19,
             "pre_lens": lambda f: de.limited_lengths([x ** 4 for x in f], 7)}]


def _dyn_hclen5():
    """the fewest code-length lengths a valid block can send: 16, 17, 18, 0 and 8 (with four, no length but 0 can be
    written and there is no end-of-block code): 255 literals and the end of block at 8 bits, no distance code"""
    lit = [8] * 255 + [0, 8]
    rnd = random.Random(12)
    return [{"type": "dynamic", "tokens": list(_rnd_bytes(rnd, 5000, bytes(range(255)))), "lit_lens": lit, "dist_lens": [0]}]


def _dyn_single_distance():
    """HDIST 1 with one 1-bit code (distance 1 only): runs of quality values"""
    rnd = random.Random(13)
    q = bytearray()
    while len(q) < 50_000:
        q += bytes([rnd.choice(b"?5+")]) * rnd.randrange(1, 80)
    return [{"type": "dynamic", "tokens": de.tokenize(bytes(q), window=1)}]


def _dyn_dna_runs18():
    """a 4-letter alphabet: 18 runs of 138 zero lengths"""
    rnd = random.Random(14)
    data = _rnd_bytes(rnd, 40_000, b"ACGT")
    return [{"type": "dynamic", "tokens": de.tokenize(data)}]


def _mixed(seed, pad):
    rnd = random.Random(seed)
    parts = [_rnd_bytes(rnd, 4000, b"ACGTN"), _rnd_bytes(rnd, 3000, b"ACGT"), _rnd_bytes(rnd, 5000, b"!#$%&'()*+")]
    d0, d1, d2 = parts
    return [{"type": "dynamic", "tokens": de.tokenize(d0), "combined": True}, {"type": "stored", "data": b"", "pad": pad},
            {"type": "fixed", "tokens": de.tokenize(d0 + d1, len(d0))},
            {"type": "dynamic", "tokens": de.tokenize(d0 + d1 + d2, len(d0) + len(d1)), "skew": True, "hlit": 286},
            {"type": "stored", "data": d2[:1000], "pad": pad}, {"type": "fixed", "tokens": [(258, 4321), (17, 2)] + _tail()}]


STREAMS = {
    "fixed_every_length_code": _fixed_lengths,
    "fixed_every_distance_code": _fixed_distances,
    "fixed_overlapping_copies": _fixed_overlaps,
    "stored_empty_first_middle_last": _stored_empty_everywhere,
    "stored_65535_plus_1": _stored_full,
    "stored_after_fixed_padding_ones": lambda: _stored_after_fixed(0x7f),
    "dynamic_literal_only_hlit257": _dyn_literal_only_257,
    "dynamic_hlit286_hdist30_run18_across": _dyn_286_30_crossing18,
    "dynamic_run16_across": _dyn_crossing16,
    "dynamic_15_bit_codes": _dyn_long_codes,
    "dynamic_7_bit_precode_hclen19": _dyn_precode7_hclen19,
    "dynamic_hclen5": _dyn_hclen5,
    "dynamic_single_distance_code": _dyn_single_distance,
    "dynamic_run18_138": _dyn_dna_runs18,
    "mixed_blocks": lambda: _mixed(15, 0),
    "mixed_blocks_padding_ones": lambda: _mixed(16, 0x55),
}

_cache = {}


def stream(name):
    """-> (compressed, bytes, census); the bytes are zlib's"""
    if name not in _cache:
        comp, data, census = de.encode(STREAMS[name]())
        assert len(data) <= 65536, (name, len(data))
        assert zlib.decompress(comp, -15) == data, name
        _cache[name] = (comp, data, census)
    return _cache[name]


# what the list as a whole must contain; a change that drops one of them fails test_census
REQUIRED = (
    ["stored_empty_first", "stored_empty_middle", "stored_empty_last", "stored_65535", "stored_pad_nonzero"]
    + ["fixed.len_%d_%s" % (s, m) for s in range(257, 286) for m in ("min", "max")]
    + ["fixed.dist_%d_%s" % (c, m) for c in range(30) for m in ("min", "max")]
    + ["fixed.dist_32768"]
    + ["fixed.copy_d%d_l%d" % (d, n) for d in range(1, 18) for n in (3, 15, 16, 17, 258)]
    + ["match_in_last_320_out", "match_in_last_16_in"]
    + ["hlit_257", "hlit_286", "hdist_1_empty", "hdist_1_len1", "hdist_30", "hclen_5", "hclen_19"]
    + ["dynamic.ll_len_15", "dynamic.dist_len_15"] + ["dynamic.dist_len_%d" % l for l in range(9, 16)]
    + ["precode_max_7", "rle16_cross", "rle18_cross", "rle18_138", "combined_rle", "split_rle"]
    + ["dist_codes_none", "dist_codes_single", "dynamic_stored_empty_fixed_dynamic"]
)


def test_census():
    total = sum((stream(n)[2] for n in STREAMS), start=collections.Counter())
    missing = [k for k in REQUIRED if not total[k]]
    assert not missing, missing


@pytest.mark.parametrize("name", sorted(STREAMS))
def test_host_decoder_alone(name):
    comp, data, _ = stream(name)
    rc, got = ti._inflate(comp, len(data))
    assert rc == 0 and got == data


@pytest.mark.parametrize("name", sorted(STREAMS))
def test_host_decoder_two_streams(name):
    names = sorted(STREAMS)
    other = names[(names.index(name) + 1) % len(names)]
    (c0, d0, _), (c1, d1, _) = stream(name), stream(other)
    for (ca, da), (cb, db) in (((c0, d0), (c1, d1)), ((c1, d1), (c0, d0))):
        rc, ga, gb = ti._inflate2(ca, len(da), cb, len(db))
        assert rc == 0 and ga == da and gb == db, other


def _e_crc():
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "himut_b200", "csrc", "bamerr.h")).read()
    names = re.findall(r"\b(E_[A-Z_]+)\b", hdr[hdr.index("enum {"):hdr.index("};")])
    return names.index("E_CRC") + 1  # E_CS_TOKEN = 1, then in order


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(STREAMS))
def test_device_decoder(ctx, name):
    comp, data, _ = stream(name)
    crc = zlib.crc32(data)
    rc, got = ctx.inflate_test(comp, len(data), crc)
    assert rc == 0 and got == data
    assert ctx.inflate_test(comp, len(data), crc ^ 1)[0] == _e_crc()
