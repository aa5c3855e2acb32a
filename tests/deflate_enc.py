"""A small raw DEFLATE (RFC 1951) encoder for tests, in plain Python.

zlib's encoder never writes several constructs that other BAM writers (libdeflate, ISA-L) do: code-length runs that
cross from the literal/length lengths into the distance lengths, header counts at their extremes, codes of 13-15 bits
the data uses, empty stored blocks between compressed ones, non-zero padding before a stored block.  This encoder
writes them on request, so that the decoders can be tested on them; zlib.decompress stays the judge of validity.

    encode(blocks) -> (compressed bytes, output bytes, census)

blocks: a list of dicts, BFINAL set on the last one only:
    {"type": "stored", "data": bytes, "pad": bits written before the byte alignment (default 0)}
    {"type": "fixed", "tokens": [...]}
    {"type": "dynamic", "tokens": [...], and optionally
        "lit_lens" / "dist_lens": code lengths (default: length-limited Huffman lengths of the tokens' symbols),
        "limit": the bound of those default lengths (15), "skew": square the counts first (longer codes),
        "hlit" / "hdist" / "hclen": the header counts (default: as few as the lengths need),
        "pre_lens": the 19 code-length code lengths, or a function of the 19 symbol counts that returns them
                    (default: Huffman lengths of the run-length symbols, <= 7 bits),
        "combined": run-length code the two length lists as one sequence (runs may cross the boundary) instead of
                    one list after the other}
A token is a literal (int 0-255) or a match (length 3-258, distance 1-32768); matches may reach into earlier blocks.
The census counts the constructs the stream contains (key -> count): header counts, code lengths used, run-length
codes and whether they cross, every length / distance symbol at its smallest and largest extra value, where matches
sit relative to the end of the input and the output.
"""
import collections

LEN_BASE = (3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258)
LEN_EXTRA = (0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0)
DIST_BASE = (1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
             6145, 8193, 12289, 16385, 24577)
DIST_EXTRA = (0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13)
PRE_ORDER = (16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15)
FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_DIST = [5] * 30


def len_symbol(n):
    """match length -> (symbol 257-285, extra bits, extra value); 258 is always 285 (not 284 + 31)"""
    if not 3 <= n <= 258:
        raise ValueError("length %d" % n)
    if n == 258:
        return 285, 0, 0
    k = max(i for i in range(28) if LEN_BASE[i] <= n)
    return 257 + k, LEN_EXTRA[k], n - LEN_BASE[k]


def dist_symbol(d):
    if not 1 <= d <= 32768:
        raise ValueError("distance %d" % d)
    k = max(i for i in range(30) if DIST_BASE[i] <= d)
    return k, DIST_EXTRA[k], d - DIST_BASE[k]


def canonical(lens):
    """RFC 1951 3.2.2: code of each symbol (None for length 0); ValueError when over-subscribed"""
    count = collections.Counter(l for l in lens if l)
    left = 1
    for l in range(1, 16):
        left = 2 * left - count[l]
        if left < 0:
            raise ValueError("over-subscribed code")
    code, nxt = 0, {}
    for l in range(1, 16):
        code = (code + count[l - 1]) << 1 if l > 1 else 0
        nxt[l] = code
    out = []
    for l in lens:
        if l:
            out.append(nxt[l])
            nxt[l] += 1
        else:
            out.append(None)
    return out


def complete(lens):
    return sum(2 ** (15 - l) for l in lens if l) == 2 ** 15


def limited_lengths(freqs, limit):
    """Huffman code lengths of at most `limit` bits (package-merge); symbols of count 0 get none; one symbol gets 1"""
    leaves = sorted((f, (s,)) for s, f in enumerate(freqs) if f > 0)
    lens = [0] * len(freqs)
    if len(leaves) == 1:
        lens[leaves[0][1][0]] = 1
        return lens
    if len(leaves) > 2 ** limit:
        raise ValueError("too many symbols for %d bits" % limit)
    cur = list(leaves)
    for _ in range(limit - 1):
        packages = [(cur[i][0] + cur[i + 1][0], cur[i][1] + cur[i + 1][1]) for i in range(0, len(cur) - 1, 2)]
        cur = sorted(leaves + packages, key=lambda x: x[0])
    for _f, syms in cur[:2 * len(leaves) - 2]:
        for s in syms:
            lens[s] += 1
    return lens


def chain_lengths(order, n):
    """a complete code over len(order) symbols of lengths 1, 2, ..., k - 1, k - 1 (k = len(order)) in that order"""
    lens = [0] * n
    k = len(order)
    for i, s in enumerate(order):
        lens[s] = min(i + 1, k - 1)
    return lens


def rle(lens):
    """code-length symbols of one sequence: [(symbol, extra bits, extra value, first index, repeat)]"""
    out, i, n = [], 0, len(lens)
    while i < n:
        v = lens[i]
        run = 1
        while i + run < n and lens[i + run] == v:
            run += 1
        if v == 0:
            left = run
            while left >= 11:
                r = min(left, 138)
                out.append((18, 7, r - 11, i + run - left, r))
                left -= r
            if left >= 3:
                out.append((17, 3, left - 3, i + run - left, left))
                left = 0
            for _ in range(left):
                out.append((0, 0, 0, i + run - left, 1))
                left -= 1
        else:
            out.append((v, 0, 0, i, 1))
            left = run - 1
            while left >= 3:
                r = min(left, 6)
                out.append((16, 2, r - 3, i + run - left, r))
                left -= r
            for _ in range(left):
                out.append((v, 0, 0, i + run - left, 1))
                left -= 1
        i += run
    return out


class BitWriter:
    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    @property
    def bitpos(self):
        return 8 * len(self.out) + self.n

    def put(self, value, nbits):
        self.acc |= (value & ((1 << nbits) - 1)) << self.n
        self.n += nbits
        while self.n >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.n -= 8

    def code(self, code, length):  # Huffman codes go most significant bit first
        self.put(int(format(code, "0%db" % length)[::-1], 2), length)

    def align(self, pad):
        k = (8 - self.n) % 8
        self.put(pad, k)
        return k

    def finish(self):
        if self.n:
            self.out.append(self.acc & 255)
            self.acc, self.n = 0, 0
        return bytes(self.out)


def tokenize(data, start=0, window=32768, max_len=258):
    """greedy LZ77 of data[start:] (matches may reach back into data[:start]) -> tokens"""
    heads = {}
    for p in range(max(0, start - window), start):
        heads[data[p:p + 3]] = p
    out, p, n = [], start, len(data)
    while p < n:
        key = data[p:p + 3]
        q = heads.get(key)
        heads[key] = p
        if q is not None and len(key) == 3 and p - q <= window:
            m = 3
            while m < max_len and p + m < n and data[q + m] == data[p + m]:
                m += 1
            out.append((m, p - q))
            for k in range(p + 1, p + m):
                heads[data[k:k + 3]] = k
            p += m
        else:
            out.append(data[p])
            p += 1
    return out


def _symbols(tokens):
    lit, dist = collections.Counter(), collections.Counter()
    for t in tokens:
        if isinstance(t, int):
            lit[t] += 1
        else:
            lit[len_symbol(t[0])[0]] += 1
            dist[dist_symbol(t[1])[0]] += 1
    lit[256] += 1
    return lit, dist


def _dynamic_header(w, blk, lit_lens, dist_lens, census):
    hlit = blk.get("hlit") or max(257, max(i for i, l in enumerate(lit_lens) if l) + 1)
    nz = [i for i, l in enumerate(dist_lens) if l]
    hdist = blk.get("hdist") or max(1, (max(nz) + 1) if nz else 1)
    if any(lit_lens[hlit:]) or any(dist_lens[hdist:]) or not 257 <= hlit <= 286 or not 1 <= hdist <= 30:
        raise ValueError("HLIT %d / HDIST %d do not hold the lengths" % (hlit, hdist))
    ll, dl = list(lit_lens[:hlit]) + [0] * (hlit - len(lit_lens)), list(dist_lens[:hdist]) + [0] * (hdist - len(dist_lens))
    seq = rle(ll + dl) if blk.get("combined") else rle(ll) + [(s, b, v, i + hlit, r) for s, b, v, i, r in rle(dl)]
    f = [0] * 19
    for s, *_ in seq:
        f[s] += 1
    if sum(1 for x in f if x) == 1:  # a code-length code must be complete: give it a second symbol
        f[0 if f[0] == 0 else 8] = 1
    pre = blk.get("pre_lens") or (lambda f: limited_lengths(f, 7))
    pre = list(pre(f) if callable(pre) else pre)
    if max(pre) > 7 or not complete(pre) or any(pre[s] == 0 for s, *_ in seq):
        raise ValueError("the code-length code does not fit")
    need = max([4] + [k + 1 for k in range(19) if pre[PRE_ORDER[k]]])
    hclen = blk.get("hclen") or need
    if not need <= hclen <= 19:
        raise ValueError("HCLEN %d < %d" % (hclen, need))
    w.put(hlit - 257, 5)
    w.put(hdist - 1, 5)
    w.put(hclen - 4, 4)
    for k in range(hclen):
        w.put(pre[PRE_ORDER[k]], 3)
    pcode = canonical(pre)
    for s, b, v, i, r in seq:
        w.code(pcode[s], pre[s])
        if b:
            w.put(v, b)
        if s >= 16:
            census["rle%d" % s] += 1
            if i < hlit < i + r or (s == 16 and i == hlit):
                census["rle%d_cross" % s] += 1
            if s == 18 and r == 138:
                census["rle18_138"] += 1
    census["hlit_%d" % hlit] += 1
    census["hclen_%d" % hclen] += 1
    census["hdist_%d" % hdist] += 1
    if hdist == 1:
        census["hdist_1_%s" % ("empty" if dl[0] == 0 else "len%d" % dl[0])] += 1
    census["precode_max_%d" % max(pre)] += 1
    census["combined_rle" if blk.get("combined") else "split_rle"] += 1


def encode(blocks):
    w = BitWriter()
    out = bytearray()
    census = collections.Counter()
    matches = []  # (output position, input bit position) of every match
    kinds = []
    for bi, blk in enumerate(blocks):
        last = bi == len(blocks) - 1
        w.put(1 if last else 0, 1)
        t = blk["type"]
        if t == "stored":
            data = bytes(blk["data"])
            if len(data) > 65535:
                raise ValueError("stored block of %d bytes" % len(data))
            w.put(0, 2)
            pad = blk.get("pad", 0)
            k = w.align(pad)
            if pad & ((1 << k) - 1):
                census["stored_pad_nonzero"] += 1
            w.put(len(data), 16)
            w.put(len(data) ^ 0xffff, 16)
            for b in data:
                w.put(b, 8)
            out += data
            census["stored"] += 1
            if not data:
                census["stored_empty_%s" % ("first" if bi == 0 else "last" if last else "middle")] += 1
            if len(data) == 65535:
                census["stored_65535"] += 1
            kinds.append("stored_empty" if not data else "stored")
            continue
        tokens = blk["tokens"]
        if t == "fixed":
            w.put(1, 2)
            lit_lens, dist_lens = FIXED_LIT, FIXED_DIST
        elif t == "dynamic":
            w.put(2, 2)
            lf, df = _symbols(tokens)
            lit_lens = blk.get("lit_lens")
            if lit_lens is None:
                f = [lf[s] ** (3 if blk.get("skew") else 1) for s in range(286)]
                lit_lens = limited_lengths(f, blk.get("limit", 15))
            dist_lens = blk.get("dist_lens")
            if dist_lens is None:
                dist_lens = limited_lengths([df[s] for s in range(30)], blk.get("limit", 15)) if df else [0]
            for name, lens, used in (("literal/length", lit_lens, lf), ("distance", dist_lens, df)):
                if any(s >= len(lens) or not lens[s] for s in used):
                    raise ValueError("a used %s symbol has no code" % name)
                nz = [l for l in lens if l]
                if nz and not complete(lens) and nz != [1]:  # zlib accepts one incomplete code: a single 1-bit code
                    raise ValueError("incomplete %s code" % name)
            _dynamic_header(w, blk, lit_lens, dist_lens, census)
            nz = [l for l in dist_lens if l]
            census["dist_codes_%s" % ("none" if not nz else "single" if len(nz) == 1 else "many")] += 1
        else:
            raise ValueError(t)
        lcode, dcode = canonical(lit_lens), canonical(list(dist_lens) + [0] * (30 - len(dist_lens)))
        for tok in tokens:
            if isinstance(tok, int):
                w.code(lcode[tok], lit_lens[tok])
                out.append(tok)
                census["%s.ll_len_%d" % (t, lit_lens[tok])] += 1
                continue
            n, d = tok
            if d > len(out):
                raise ValueError("distance %d before the start of the output" % d)
            matches.append((len(out), w.bitpos))
            s, eb, ev = len_symbol(n)
            w.code(lcode[s], lit_lens[s])
            w.put(ev, eb)
            ds, deb, dev = dist_symbol(d)
            w.code(dcode[ds], dist_lens[ds])
            w.put(dev, deb)
            for k in range(n):
                out.append(out[-d])
            census["%s.ll_len_%d" % (t, lit_lens[s])] += 1
            census["%s.dist_len_%d" % (t, dist_lens[ds])] += 1
            for key, x, bits in (("len_%d" % s, ev, eb), ("dist_%d" % ds, dev, deb)):
                if x == 0:
                    census["%s.%s_min" % (t, key)] += 1
                if x == (1 << bits) - 1 - (key == "len_284"):  # 284 + 31 (= 258) is not written
                    census["%s.%s_max" % (t, key)] += 1
            if d == 32768:
                census["%s.dist_32768" % t] += 1
            if d <= 17 and n in (3, 15, 16, 17, 258):
                census["%s.copy_d%d_l%d" % (t, d, n)] += 1
        w.code(lcode[256], lit_lens[256])
        census[t] += 1
        kinds.append(t)
    comp = w.finish()
    for opos, bpos in matches:
        if opos >= len(out) - 320:
            census["match_in_last_320_out"] += 1
        if bpos >= 8 * (len(comp) - 16):
            census["match_in_last_16_in"] += 1
    for i in range(len(kinds) - 3):
        if kinds[i:i + 4] == ["dynamic", "stored_empty", "fixed", "dynamic"]:
            census["dynamic_stored_empty_fixed_dynamic"] += 1
    census["blocks_%d" % len(blocks)] += 1
    return comp, bytes(out), census
