#!/usr/bin/env python
"""Fuzzing session: the native BAM decoder (csrc/bamdec.c) against the Python specification (bamio.py + pack.py) on
adversarial batches (dense substitutions / indels, N bases, soft clips, secondary records, duplicate names) written
to multi-contig BAM files: random windows, thread counts, with and without the base stream — packed batches must be
equal byte for byte, the window pre-pass must return the same read lengths.
    python tools/fuzz_bamdec_vs_spec.py 0 200 [--tags md | md_eqx]
--tags: the files carry CIGAR + MD:Z instead of cs:Z (the decoders' MD path; the Python side reads them with
pack.parse_md).
(400 seeds x 6 windows on 2026-10-18: no mismatch.)"""
import os
import random
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import cases  # noqa: E402
from himut_b200 import bamdec, bamio, pack  # noqa: E402


def same(a, b, skip=()):
    for name, _ in a._FIELDS:
        if name in skip:
            continue
        x, y = getattr(a, name), getattr(b, name)
        if x.shape != y.shape or not np.array_equal(x, y):
            return name
    return None


def main():
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("lo", type=int)
    ap.add_argument("hi", type=int)
    ap.add_argument("--tags", default="cs", choices=["cs", "md", "md_eqx"])
    args = ap.parse_args()
    lo, hi = args.lo, args.hi
    bad = 0
    with tempfile.TemporaryDirectory() as tmp:
        for seed in range(lo, hi):
            rnd = random.Random(seed * 13 + 5)
            contigs = []
            for k in range(rnd.choice([1, 2, 3])):
                n = rnd.choice([1500, 6000, 30000])
                batch, _ref = cases.adversarial_batch(seed * 10 + k, contig_len=n, n_reads=rnd.choice([0, 40, 200]) if k else rnd.choice([40, 200]),
                                                      max_len=rnd.choice([300, 2000, 9000]))
                contigs.append(("c%d" % k, n, batch))
            path = os.path.join(tmp, "f%d.bam" % seed)
            bamio.write_batches_bam(path, contigs, tags=args.tags)
            nb = bamdec.NativeBam(path, threads=rnd.choice([1, 2, 5]))
            rd = bamio.BamReader(path)
            qnames = {}
            for _ in range(6):
                c, n, _b = rnd.choice(contigs)
                a = rnd.randrange(0, n)
                e = min(n, a + rnd.choice([1, 50, 1000, n]))
                bb = pack.BatchBuilder()
                bb.qnames = qnames
                want = bamio.read_batch(rd, c, a, e, builder=bb)
                seq = rnd.random() < 0.5
                got = nb.read_batch(c, a, e, seq=seq)
                why = same(got, want, skip=() if seq else ("seq", "seq_off"))
                if why:
                    bad += 1
                    print("seed", seed, c, a, e, "seq" if seq else "noseq", "field", why)
                qs = nb.window_qlens(c, a, e)
                exp = [len(r.query_sequence) for r in rd.fetch(c, a, e) if r.mapping_quality > 0 and r.has_tag("tp") and r.get_tag("tp") == "P"]
                if qs.tolist() != exp:
                    bad += 1
                    print("seed", seed, c, a, e, "window_qlens", qs.size, len(exp))
            nb.close(); rd.close()
            os.unlink(path); os.unlink(path + ".bai")
    print("seeds", lo, hi, "mismatches", bad)
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
