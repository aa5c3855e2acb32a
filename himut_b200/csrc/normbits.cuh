// normbits.cuh — the callable-base half of `himut normcounts` as bit vectors (sm_100a): the integer pass in front of the
// exact pass (normfast.cuh).
//
// The reference asks two things of every aligned base (normcounts.py:65-110, 292-314): "does this read count here"
// (matched base, BQ >= min_bq, no mismatch within the window of its block, not trimmed) and "what does the pileup
// column look like" (gtlib.get_germ_gt over every base of the column).  At a *pure* position — every primary read that
// covers it shows the FASTA base through a plain cs match — the second question has a certified answer that needs the
// depth n and a lower bound of the column's quality sum only (NormCert, himut_b200.cu).  And a lower bound is at hand
// without touching a single quality byte again: every counted base has BQ >= min_bq, every other base has BQ >= 1, so
//     sum BQ  >=  min_bq * callable + (n - callable).
// So each read is turned ONCE, by the warp that streams its qualities anyway, into one bit per reference position
// ("this read counts here"), and the per-position work becomes adding bit vectors:
//
//   k_ref_pack    the contig as 2-bit codes + the trinucleotide bin of every position (once per reference).
//   k_norm_prep   one warp per read (replaces k_read_scan on this path and does all it does): cs op prefix scan,
//                 mismatch list, identity / QV gates, the whole-read quality sum — and, from the same 16-byte quality
//                 words, the bit "BQ >= min_bq" per query base.  Then per 32 reference positions of the read: the
//                 bits of the match runs moved to reference coordinates, minus trimmed and window-blocked positions
//                 (get_trimmed_range / get_mismatch_range, bamlib.py:222-258) -> cal[read][word].  Positions where the
//                 read is anything but a plain match of the FASTA base (substitution, deletion, the base an insertion
//                 precedes, a match run base that differs from the FASTA, BQ 0, op lists too long to stage) are set in
//                 a per-contig `impure` bitmap.
//   k_norm_bits   one warp per 1024 reference positions, lane = 32 positions.  The covering reads in file order: the
//                 coverage word and the cal word of each are added into bit-sliced counters (carry-save adders, three
//                 logic ops per read and counter); depth, callable count and haplotype tallies of all 32 positions of
//                 a lane never leave 8 + 8 (+ 16) registers.  Then, bit-parallel: certified -> the cascade's depth /
//                 ref-count gates and the 33-bin tallies (normcounts.py:317-400); impure or not certified -> the site
//                 list of the exact pass (k_norm_entries_bits below, k_norm_reduce in normfast.cuh), which evaluates the
//                 position with the reference's own ordered fp64 arithmetic.  Both passes add into the same tallies.
//
// The verdict at a certified position is the exact verdict (tests/test_norm_cert.py holds the bound against the
// reference's gtlib); everything else is evaluated exactly, so the result is bit-identical to genotyping every column.
#pragma once
#include "normfast.cuh"

#define NB_OPS 192u                 // ops of a read staged in shared memory (more: the read's span goes to the exact pass)
#define NB_SEG 4096u                // query bases a warp holds in shared memory at a time (a read is walked segment by segment)
#define NB_PREP_WARPS 4
#define NB_SPAN 1024                // reference positions per warp of k_norm_bits
#define NB_BITS_WARPS 4

struct __align__(16) PrepWarp {
  uint32_t qg[NB_SEG / 32 + 4];     // bit q: BQ of the segment's query base q >= min_bq (then: "counts")
  uint32_t sq[NB_SEG / 16 + 4];     // the segment's 2-bit bases
  uint32_t rf[NB_SEG / 16 + 16];    // the 2-bit reference under the segment (a segment with long deletions reads ref2 directly)
  uint32_t w[NB_OPS], t[NB_OPS + 1], q[NB_OPS + 1]; // t / q[k + 1] = where op k ends (t / q[nops]: the read's totals)
  int32_t mm[NB_OPS];               // op index of every entry of the mismatch list
  uint32_t mr[NB_OPS];              // op index of every match run, ascending
};

// ============================================================================ k_ref_pack
// ref2: 16 positions per word, HM base codes (A 0, T 1, G 2, C 3; anything else 0); tri8: get_tri_context bin
// (normcounts.py:49-62) of a position whose base is upper-case A/C/G/T, else 255 (normcounts.py:320 skips it).
// Both cover n_pos >= ref_len positions (multiple of 32); past the reference: 0 / 255.
__global__ void __launch_bounds__(256) k_ref_pack(const uint8_t* refseq, uint64_t ref_len, uint64_t n_pos, uint32_t* ref2, uint8_t* tri8) {
  const uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; // one thread per 16 positions
  if (w * 16 >= n_pos) return;
  uint32_t code = 0;
  uint32_t tb[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
#pragma unroll
  for (int k = 0; k < 16; k++) {
    const uint64_t pos = w * 16 + k;
    if (pos >= ref_len) continue;
    const uint8_t ch = __ldg(refseq + pos);
    const int c = ch == 'A' ? 0 : ch == 'T' ? 1 : ch == 'G' ? 2 : ch == 'C' ? 3 : -1;
    if (c < 0) continue;
    code |= (uint32_t)c << (2 * k);
    const uint32_t tri = (uint32_t)tri_bin_dev(refseq, ref_len, (int64_t)pos);
    tb[k >> 2] = (tb[k >> 2] & ~(0xffu << (8 * (k & 3)))) | (tri << (8 * (k & 3)));
  }
  ref2[w] = code;
  reinterpret_cast<uint4*>(tri8)[w] = make_uint4(tb[0], tb[1], tb[2], tb[3]);
}

__device__ __forceinline__ uint32_t spread4(uint32_t nib) { return (nib * 0x00204081u) & 0x01010101u; } // bit k -> bit 8k

// the k lowest bits (k <= 0: none, k >= 32: all): one BMSK with its width clamped to [0, 32] (k_norm_prep 1.25 -> 1.20 ms,
// k_norm_bits 0.28 -> 0.27 ms against the compare-and-shift form, NB_NO_BMSK)
__device__ __forceinline__ uint32_t low_mask(int k) {
#ifndef NB_NO_BMSK
  uint32_t m;
  asm("bmsk.clamp.b32 %0, 0, %1;" : "=r"(m) : "r"((uint32_t)max(k, 0)));
  return m;
#else
  return k >= 32 ? 0xffffffffu : (k <= 0 ? 0u : ((1u << k) - 1u));
#endif
}
__device__ __forceinline__ void mark_impure(uint32_t* impure, uint64_t imp_words, int64_t pos) {
  if (pos >= 0 && (uint64_t)(pos >> 5) < imp_words) atomicOr(impure + (pos >> 5), 1u << (pos & 31));
}
__device__ __forceinline__ void mark_impure_range(uint32_t* impure, uint64_t imp_words, int64_t lo, int64_t hi) { // [lo, hi)
  if (lo < 0) lo = 0;
  while (lo < hi) {
    const int64_t wi = lo >> 5;
    const int b0 = (int)(lo & 31), n = (int)min((int64_t)(32 - b0), hi - lo);
    if ((uint64_t)wi < imp_words) atomicOr(impure + wi, low_mask(n) << b0);
    lo += n;
  }
}

// ============================================================================ k_norm_prep
// One warp per read.  Writes everything k_read_scan writes (op_t, op_q, mm_pos, the totals, the gate byte), plus the
// read's cal words at calw[cw_off[r] ...) — word j holds reference positions 32 * ((tstart >> 5) + j) ... + 31 — and
// the read's contribution to the impure bitmap.  Secondary records are skipped by every consumer: they get neither.
//
// The bits live in QUERY coordinates as long as possible: "BQ >= min_bq" comes out of the quality words in query
// order; the trimmed ends are two masks; the mismatch window of a block (get_mismatch_range is anchored at the block's
// first base, so the window of a mismatch differs from block to block) clears, per (mismatch, nearby block), one range
// of query positions.  What is left is moved to reference coordinates run by run: a funnel shift per 32 positions.
__global__ void __launch_bounds__(32 * NB_PREP_WARPS, 8) k_norm_prep(DevBatch b, DevParams p, const uint32_t* ref2, const uint32_t* cw_off,
                                                                   uint32_t* calw, uint32_t* impure, uint64_t imp_words,
                                                                   const uint16_t* mask16, const uint8_t* exc_minmax,
                                                                   uint32_t modal, uint32_t* sdiff,
                                                                   uint8_t* cal_ok) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= b.n_reads) return;
  PrepWarp* S = reinterpret_cast<PrepWarp*>(smem_raw) + (threadIdx.x >> 5);
  const uint64_t o0 = __ldg(b.op_off + r);
  const uint32_t nops = __ldg(b.n_ops + r);
  const int32_t ts = __ldg(b.tstart + r), te = __ldg(b.tend + r);
  const int32_t qlen = __ldg(b.qlen + r);
  const uint32_t qstart = (uint32_t)__ldg(b.qstart + r);
  const bool primary = !(__ldg(b.flags + r) & HM_READ_SECONDARY);
  const uint8_t* bq = b.bq + __ldg(b.bq_off + r);

  // ---- phase 1: op prefix scan (k_read_scan), ops staged, non-match ops -> impure
  uint32_t t_carry = 0, q_carry = qstart;
  int mm_base = 0, nm = 0, ns = 0, il = 0, dl = 0;
  uint32_t n_runs = 0;
  for (uint32_t base = 0; base < nops; base += 32) {
    const uint32_t k = base + lane;
    const bool valid = k < nops;
    const uint32_t w = valid ? __ldg(b.ops + o0 + k) : 0u;
    const uint32_t kind = w & 3u, v = w >> 2;
    const uint32_t rl = (uint32_t)op_ref_len(w), al = (uint32_t)op_qry_len(w);
    uint32_t rs = rl, qs = al;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t a = __shfl_up_sync(HM_FULL, rs, d), c = __shfl_up_sync(HM_FULL, qs, d);
      if (lane >= d) { rs += a; qs += c; }
    }
    const uint32_t t_ex = t_carry + rs - rl, q_ex = q_carry + qs - al;
    if (valid) {
      b.op_t[o0 + k] = t_ex; b.op_q[o0 + k] = q_ex;
      if (k < NB_OPS) { S->w[k] = w; S->t[k] = t_ex; S->q[k] = q_ex; }
    }
    const bool is_mm = valid && ((kind == HM_OP_SUB && (v & 7u) != HM_BASE_N) || kind == HM_OP_INS || kind == HM_OP_DEL);
    const uint32_t bal = __ballot_sync(HM_FULL, is_mm);
    if (is_mm) {
      const uint32_t at = (uint32_t)mm_base + __popc(bal & ((1u << lane) - 1u));
      b.mm_pos[o0 + at] = ts + (int32_t)t_ex + 1;
      if (at < NB_OPS) S->mm[at] = (int32_t)k; // the op that is this entry of the list
    }
    mm_base += __popc(bal);
    {
      const bool is_run = valid && kind == HM_OP_MATCH && v != 0u;
      const uint32_t br = __ballot_sync(HM_FULL, is_run);
      if (is_run) { const uint32_t at = n_runs + __popc(br & ((1u << lane) - 1u)); if (at < NB_OPS) S->mr[at] = k; }
      n_runs += __popc(br);
    }
    if (valid) {
      if (kind == HM_OP_MATCH) nm += (int)v;
      else if (kind == HM_OP_SUB) ns += 1;
      else if (kind == HM_OP_INS) il += (int)v;
      else dl += (int)v;
      if (primary && kind != HM_OP_MATCH) { // update_allelecounts: a substituted / deleted base, or the base an insertion precedes
        const int64_t at = (int64_t)ts + t_ex;
        if (kind == HM_OP_DEL) mark_impure_range(impure, imp_words, at, at + v);
        else mark_impure(impure, imp_words, at);
      }
    }
    t_carry += __shfl_sync(HM_FULL, rs, 31);
    q_carry += __shfl_sync(HM_FULL, qs, 31);
  }
  nm = __reduce_add_sync(HM_FULL, nm);
  ns = __reduce_add_sync(HM_FULL, ns);
  il = __reduce_add_sync(HM_FULL, il);
  dl = __reduce_add_sync(HM_FULL, dl);
  if (lane == 0 && nops <= NB_OPS) { S->t[nops] = t_carry; S->q[nops] = q_carry; }
  __syncwarp();

  // ---- phases 2 and 3, one segment of NB_SEG query bases after the other (shared memory holds one segment)
  const uint32_t nw = (primary && te > ts) ? (uint32_t)(((te - 1) >> 5) - (ts >> 5) + 1) : 0u;
  uint32_t* out = calw + __ldg(cw_off + r);
  // a read whose ops this kernel cannot stage, or do not add up to its span: every position of the span is evaluated
  // by the exact pass (so is a read with a quality of 0, found below: the reference raises there)
  const bool staged = nops != 0 && nops <= NB_OPS && t_carry == (uint32_t)(te - ts);
  const bool do_bits = nw != 0 && staged;
  const uint32_t kge = (uint32_t)(128 - p.min_bq) * 0x01010101u; // byte >= min_bq  <=>  bit 7 of ((byte & 0x7f) + 128 - min_bq) | byte
  const uint4* q4 = reinterpret_cast<const uint4*>(bq);
  const uint32_t* seq32 = reinterpret_cast<const uint32_t*>(b.seq + __ldg(b.seq_off + r));
  uint16_t* qg16 = reinterpret_cast<uint16_t*>(S->qg);
  const int32_t trim_s = (int32_t)floor(__dmul_rn(p.min_trim, (double)qlen));
  const int32_t trim_e = (int32_t)ceil(__dmul_rn(__dsub_rn(1.0, p.min_trim), (double)qlen));
  const int wsz = p.mismatch_window, max_mm = p.max_mismatch_count;
  const uint32_t nmm = (uint32_t)mm_base;
  const int32_t ts_lo = ts & 31;
  // get_mismatch_range(rpos, qpos, qlen, window) with (rpos, qpos) the block's first base (normcounts.py:82,
  // bamlib.py:245-258) gives the block its (u, d); a base at read offset o counts the list entries x1 (1-based read
  // offsets) with o - u <= x1 <= o + d (normcounts.py:84-87)
  auto block_ud = [&](int32_t qk, int* u, int* d) {
    const int qs = qk - wsz, qe = qk + wsz;
    if (qs < 0) { *u = wsz + qs; *d = wsz + (-qs); }
    else if (qe > qlen) { *u = wsz + (qe - qlen); *d = qlen - qk; }
    else { *u = wsz; *d = wsz; }
  };
  // A batch that came as bitmap + exceptions (hm_bq_compact) and whose exceptions of this read all lie below min_bq:
  // "BQ >= min_bq" is the bitmap itself (or nothing, when the modal value is below min_bq too), the quality sum was
  // taken when the stream was expanded, and no quality byte is touched here.
  bool use_mask = false;
  uint32_t e_min = 255u;
  if (mask16 != nullptr && modal != 0u) {
    e_min = __ldg(exc_minmax + 2 * r);
    use_mask = (int)__ldg(exc_minmax + 2 * r + 1) < p.min_bq;
  }
  const uint64_t bq_bit0 = __ldg(b.bq_off + r); // the read's first bit in the bitmap
  uint32_t acc = 0, zacc = 0;
  int32_t o_seg = 0;               // read offset at which the current segment's reference positions begin
  uint32_t rp = 0;                 // first match run that can reach into the current segment
  // words that several match runs (or two segments) share are OR-ed into place; words no run reaches stay 0
  for (uint32_t j = (uint32_t)lane; j < nw; j += 32) out[j] = 0u;
  __syncwarp();
  for (int32_t seg0 = 0; seg0 < qlen; seg0 += (int32_t)NB_SEG) {
    if (use_mask && !do_bits) break; // nothing of this read is wanted
    const int32_t seg1 = min(seg0 + (int32_t)NB_SEG, qlen);
    // The segment owns the read offsets [o_seg, o_next): o_next = where the next segment's first base lies.
    // ks / ke: the first op that ends past query position seg0 / seg1 (op ends ascend: a count is an index)
    uint32_t ks = 0, ke = 0;
    int32_t o_next = te - ts;
    uint32_t R0 = 0;
    bool rf_staged = false;
    if (do_bits) {
      for (uint32_t base = 0; base < nops; base += 32) {
        const uint32_t k = base + (uint32_t)lane;
        const int32_t qe = k < nops ? (int32_t)S->q[k + 1] : INT32_MAX;
        ks += __popc(__ballot_sync(HM_FULL, qe <= seg0));
        ke += __popc(__ballot_sync(HM_FULL, qe <= seg1));
      }
      if (seg1 < qlen && ke < nops) {
        const uint32_t wd = S->w[ke];
        o_next = (int32_t)S->t[ke] + ((wd & 3u) == HM_OP_MATCH ? max(seg1 - (int32_t)S->q[ke], 0) : 0);
      }
      if (o_next > o_seg) { // the 2-bit reference under the segment, from a 64-position border on; loads first, then stores
        R0 = (uint32_t)((ts + o_seg) >> 6) << 2;
        const uint32_t cnt4 = ((((uint32_t)((ts + o_next - 1) >> 5) << 1) + 2u - R0) + 3u) >> 2;
        rf_staged = cnt4 <= (NB_SEG / 16 + 16) / 4;
        if (rf_staged) {
          const uint4* src = reinterpret_cast<const uint4*>(ref2 + R0);
          uint4 v[5];
#pragma unroll
          for (int u = 0; u < 5; u++) { const uint32_t i = (uint32_t)lane + 32u * u; v[u] = i < cnt4 ? __ldg(src + i) : make_uint4(0u, 0u, 0u, 0u); }
#pragma unroll
          for (int u = 0; u < 5; u++) { const uint32_t i = (uint32_t)lane + 32u * u; if (i < cnt4) reinterpret_cast<uint4*>(S->rf)[i] = v[u]; }
        }
      }
    }
    // -- phase 2: the segment's quality words once — whole-read sum (np.mean is an exact integer sum divided once),
    // one bit per base "BQ >= min_bq"; the segment's bases staged next to them
    const uint32_t i0 = (uint32_t)seg0 >> 4, i1 = ((uint32_t)seg1 + 15u) >> 4;
    auto one_word = [&](uint4 v, uint32_t i) {
      uint32_t wv[4] = {v.x, v.y, v.z, v.w}, zw[4] = {v.x, v.y, v.z, v.w};
      const uint32_t g0 = i << 4;
      uint32_t live = 0xffffu;
      if (g0 + 16u > (uint32_t)qlen) { // padding bytes are not part of the read: 0 for the sum, non-zero for the zero test
        const uint32_t keep = (uint32_t)qlen - g0; // 1 .. 15
        live = (1u << keep) - 1u;
#pragma unroll
        for (int j = 0; j < 4; j++) {
          const int kb = (int)keep - 4 * j;
          const uint32_t mk = kb >= 4 ? 0xffffffffu : kb <= 0 ? 0u : ((1u << (8 * kb)) - 1u);
          wv[j] &= mk;
          zw[j] = wv[j] | ~mk;
        }
      }
      uint32_t bits = 0;
#pragma unroll
      for (int j = 0; j < 4; j++) {
        acc = sum4(wv[j], acc);
        const uint32_t ge = (((wv[j] & 0x7f7f7f7fu) + kge) | wv[j]) & 0x80808080u; // bit 7 of each byte: BQ >= min_bq
        bits |= ((ge * 0x00204081u) >> 28) << (4 * j);                               // bits 7, 15, 23, 31 -> a nibble
        zacc |= (zw[j] - 0x01010101u) & ~zw[j];                                      // bit 7 of some byte set iff a byte of the word is 0
      }
      if (do_bits) qg16[i - i0] = (uint16_t)(bits & live);
    };
    if (use_mask) {
      // -- phase 2 without the quality bytes: the segment's bitmap words and its bases
      const uint32_t nqw = ((uint32_t)(seg1 - seg0) + 31u) >> 5;
      const uint64_t u16_0 = (bq_bit0 >> 4) + ((uint32_t)seg0 >> 4); // bq_off is a multiple of 16: the bitmap is 16-bit aligned per read
      const uint32_t* m32 = reinterpret_cast<const uint32_t*>(mask16 + (u16_0 & ~1ull));
      const uint32_t msh = (uint32_t)(u16_0 & 1ull) * 16u;
      const bool modal_counts = modal >= (uint32_t)p.min_bq;
      const uint4* s4 = reinterpret_cast<const uint4*>(seq32 + i0);
      const uint32_t n4 = (i1 - i0 + 3u) >> 2;
      uint32_t ma[NB_SEG / 1024], mb[NB_SEG / 1024];
      uint4 sv[NB_SEG / 2048];
#pragma unroll
      for (uint32_t u = 0; u < NB_SEG / 1024; u++) { // all loads first
        const uint32_t wi = (uint32_t)lane + 32u * u;
        const bool on = wi < nqw && modal_counts;
        ma[u] = on ? __ldg(m32 + wi) : 0u; mb[u] = on ? __ldg(m32 + wi + 1) : 0u;
      }
#pragma unroll
      for (uint32_t u = 0; u < NB_SEG / 2048; u++) { const uint32_t i = (uint32_t)lane + 32u * u; sv[u] = i < n4 ? __ldg(s4 + i) : make_uint4(0u, 0u, 0u, 0u); }
#pragma unroll
      for (uint32_t u = 0; u < NB_SEG / 1024; u++) {
        const uint32_t wi = (uint32_t)lane + 32u * u;
        // past the read: padding, then the next read's bits
        if (wi < nqw) S->qg[wi] = __funnelshift_r(ma[u], mb[u], msh) & low_mask(qlen - (seg0 + (int32_t)(wi * 32u)));
      }
#pragma unroll
      for (uint32_t u = 0; u < NB_SEG / 2048; u++) { const uint32_t i = (uint32_t)lane + 32u * u; if (i < n4) reinterpret_cast<uint4*>(S->sq)[i] = sv[u]; }
      __syncwarp();
    } else {
      uint32_t i = i0 + (uint32_t)lane;
      for (; i + 96 < i1; i += 128) {
        const uint4 a0 = ldg_stream16(q4 + i), a1 = ldg_stream16(q4 + i + 32), a2 = ldg_stream16(q4 + i + 64), a3 = ldg_stream16(q4 + i + 96);
        uint32_t s0 = 0, s1 = 0, s2 = 0, s3 = 0;
        if (do_bits) { s0 = __ldg(seq32 + i); s1 = __ldg(seq32 + i + 32); s2 = __ldg(seq32 + i + 64); s3 = __ldg(seq32 + i + 96); }
        one_word(a0, i); one_word(a1, i + 32); one_word(a2, i + 64); one_word(a3, i + 96);
        if (do_bits) { S->sq[i - i0] = s0; S->sq[i - i0 + 32] = s1; S->sq[i - i0 + 64] = s2; S->sq[i - i0 + 96] = s3; }
      }
      for (; i < i1; i += 32) {
        const uint4 a0 = ldg_stream16(q4 + i);
        if (do_bits) S->sq[i - i0] = __ldg(seq32 + i);
        one_word(a0, i);
      }
    }
    if (!do_bits) continue;
    { // the words the funnel shifts below may touch past the segment's last base
      const uint32_t n16 = i1 - i0;
      for (uint32_t i = (use_mask ? ((n16 + 1u) & ~1u) : n16) + (uint32_t)lane; i < ((n16 + 1u) & ~1u) + 4u; i += 32) qg16[i] = 0;
      for (uint32_t i = n16 + (uint32_t)lane; i < n16 + 3u; i += 32) S->sq[i] = 0;
    }
    __syncwarp();

    // -- phase 2b, still in query coordinates: trimmed ends and mismatch windows
    { // get_trimmed_range / is_trimmed (bamlib.py:222-242): q < trim_s or q > trim_e does not count
      const uint32_t nqw = ((uint32_t)(seg1 - seg0) + 31u) >> 5;
      for (uint32_t wi = (uint32_t)lane; wi < nqw; wi += 32) {
        const int32_t q0 = seg0 + (int32_t)(wi * 32u);
        const uint32_t keep = low_mask(trim_e + 1 - q0) & ~low_mask(trim_s - q0);
        if (keep != 0xffffffffu) S->qg[wi] &= keep;
      }
    }
    __syncwarp();
    // with max_mismatch_count = 0 a single list entry in its window blocks a base: lane = one entry of the list,
    // which clears o in [x1 - d, x1 + u] in the blocks around it (the part that lies in this segment)
#ifdef NB_X_NO_2B
    if (max_mm == 12345) {
#else
    if (max_mm == 0) {
#endif
      for (uint32_t m = (uint32_t)lane; m < nmm; m += 32) {
        const int32_t km = S->mm[m];
        const int32_t x1 = (int32_t)S->t[km] + 1;
        auto clear_in_block = [&](int32_t kk) {
          const uint32_t wd = S->w[kk];
          const int32_t tk = (int32_t)S->t[kk], len = (int32_t)(wd >> 2), qk = (int32_t)S->q[kk];
          if (qk >= seg1 || qk + len <= seg0) return;
          int u, d;
          block_ud(qk, &u, &d);
          const int32_t lo = max(x1 - d, tk), hi = min(x1 + u, tk + len - 1); // inclusive
          if (lo > hi) return;
          int32_t q0 = max(qk + (lo - tk), seg0) - seg0;
          const int32_t q1 = min(qk + (hi - tk), seg1 - 1) - seg0;
          while (q0 <= q1) {
            const int32_t wi = q0 >> 5, b0 = q0 & 31, n = min(32 - b0, q1 - q0 + 1);
            atomicAnd(&S->qg[wi], ~(low_mask(n) << b0));
            q0 += n;
          }
        };
        for (int32_t kk = km + 1; kk < (int32_t)nops; kk++) { // blocks after the entry
          if ((int32_t)S->t[kk] > x1 + 2 * wsz) break;
          if ((S->w[kk] & 3u) == HM_OP_MATCH) clear_in_block(kk);
        }
        for (int32_t kk = km - 1; kk >= 0; kk--) {            // blocks before it
          const uint32_t wd = S->w[kk];
          if ((int32_t)S->t[kk + 1] - 1 < x1 - 2 * wsz) break;
          if ((wd & 3u) == HM_OP_MATCH) clear_in_block(kk);
        }
      }
      __syncwarp();
    }

    // -- phase 3: the bits of the match runs to reference coordinates; the bases of the runs against the FASTA.
    // Run by run (warp-uniform), lanes = the run's 32-position words.
#ifdef NB_X_NO_P3
    if (o_next > -5) { o_seg = o_next; __syncwarp(); continue; }
#endif
    while (rp < n_runs && S->mr[rp] < ks) rp++; // first match run of the segment (runs ascend with the segments)
    for (uint32_t ri = rp; ri < n_runs && o_next > o_seg; ri++) {
      const uint32_t k = S->mr[ri];
      const int32_t tk = (int32_t)S->t[k];
      if (tk >= o_next) break;
      const int32_t lo_s = max(tk, o_seg), hi_s = min((int32_t)S->t[k + 1], o_next); // the run's part in this segment
      if (lo_s >= hi_s) continue;
      const int32_t qk = (int32_t)S->q[k];
      const uint32_t jf = (uint32_t)(lo_s + ts_lo) >> 5, jl = (uint32_t)(hi_s - 1 + ts_lo) >> 5;
      for (uint32_t j = jf + (uint32_t)lane; j <= jl; j += 32) {
        const int32_t a = (int32_t)(j * 32u) - ts_lo; // read offset of this word's first position
        const int32_t lo = max(a, lo_s), hi = min(a + 32, hi_s);
        const int nb = hi - lo, sh = lo - a;
        const int32_t qb = qk + (lo - tk) - seg0; // query position of the first base, in the segment
        uint32_t g = __funnelshift_r(S->qg[qb >> 5], S->qg[(qb >> 5) + 1], (uint32_t)(qb & 31)) & low_mask(nb);
        if (max_mm != 0 && g) { // general threshold: count the list entries in the window of every candidate base
          int u, d;
          block_ud(qk, &u, &d);
          uint32_t todo = g;
          while (todo) {
            const int bit = __ffs(todo) - 1;
            todo &= todo - 1;
            const int32_t o = lo + bit;
            int cnt = 0;
            for (uint32_t m = 0; m < nmm; m++) {
              const int32_t x1 = (int32_t)S->t[S->mm[m]] + 1;
              if (x1 > o + d) break;
              cnt += (x1 >= o - u);
            }
            if (cnt > max_mm) g &= ~(1u << bit);
          }
        }
        if (nb == 32) out[j] = g;                    // the word is this run's alone
        else if (g) atomicOr(out + j, g << sh);
#ifndef NB_X_NO_SEQ
        { // a cs match that is not the FASTA's base makes the column impure
          const uint64_t W = (uint64_t)(ts >> 5) + j;
          uint2 rf;
          if (rf_staged) rf = *reinterpret_cast<const uint2*>(&S->rf[2u * (uint32_t)W - R0]);
          else rf = __ldg(reinterpret_cast<const uint2*>(ref2) + W);
          const unsigned long long rf64 = (unsigned long long)rf.x | ((unsigned long long)rf.y << 32);
          const uint32_t s = (uint32_t)qb >> 4, bsh = 2u * ((uint32_t)qb & 15u);
          const uint32_t w0 = S->sq[s], w1 = S->sq[s + 1], w2 = S->sq[s + 2];
          const unsigned long long rd = (unsigned long long)__funnelshift_r(w0, w1, bsh) | ((unsigned long long)__funnelshift_r(w1, w2, bsh) << 32);
          const unsigned long long rng = (nb >= 32 ? ~0ull : ((1ull << (2 * nb)) - 1ull)) << (2 * sh);
          const unsigned long long x = ((rd << (2 * sh)) ^ rf64) & rng;
          if (x) {
            unsigned long long dd = (x | (x >> 1)) & 0x5555555555555555ull;
            while (dd) {
              const int bit = __ffsll((long long)dd) - 1;
              dd &= dd - 1;
              mark_impure(impure, imp_words, (int64_t)(W << 5) + (bit >> 1));
              mark_impure(sdiff, imp_words, (int64_t)(W << 5) + (bit >> 1)); // the exact pass reads this read's base here
            }
          }
        }
#endif
      }
    }
    o_seg = o_next;
    __syncwarp(); // shared memory is refilled by the next segment
  }
  unsigned long long tot = acc;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) tot += __shfl_xor_sync(HM_FULL, tot, d);
  bool has_zero = __any_sync(HM_FULL, (zacc & 0x80808080u) != 0u);
  if (use_mask) { tot = b.bq_total[r]; has_zero = e_min == 0u; } // the resident sum (the bytes were not all read)
  if (lane == 0) {
    cal_ok[r] = do_bits ? 1 : 0; // the read's cal words are what update_tri2count counts (the exact pass takes them from there)
    b.bq_total[r] = tot;
    b.n_match[r] = nm; b.n_sub[r] = ns; b.ins_len[r] = il; b.del_len[r] = dl; b.n_mm[r] = mm_base;
    bool ok = true; // caller.py:310-317 / normcounts.py:302-309, in order
    const double qv = __ddiv_rn((double)tot, (double)qlen);
    if (qv < (double)p.min_qv) ok = false;
    if ((int)__ldg(b.mapq + r) < p.min_mapq) ok = false;
    const double ident = __ddiv_rn((double)nm, (double)(nm + ns + il + dl));
    if (ident < p.min_sequence_identity) ok = false;
    if (!(p.qlen_lower_limit < qlen && qlen < p.qlen_upper_limit)) ok = false;
    b.gate[r] = ok ? 1 : 0;
  }
  if (nw != 0 && (!staged || has_zero)) {
    const int64_t per = ((int64_t)(te - ts) + 31) / 32; // every lane a piece of [ts, te)
    mark_impure_range(impure, imp_words, (int64_t)ts + per * lane, min((int64_t)te, (int64_t)ts + per * (lane + 1)));
  }
}

// ============================================================================ k_norm_entries_bits
// The exact pass's gather, one warp per (chunk, read) pair as k_site_entries_by_read (kernels.cuh) does it for `call`.
// It stages the read's op arrays in shared memory and serves every listed site of the chunk the read covers; `keys` is
// in (chunk, position) order and [s0, s0 + nb) is the slice of it this launch fills (entries are slice relative).
// "Is this base counted by update_tri2count" is the read's cal bit (no window / trim arithmetic), the base of a match
// run is the FASTA's unless k_norm_prep saw it differ (sdiff), and on a compact upload the quality is the modal value wherever the bitmap says so — the byte
// stream is touched for the exceptions only.  Reads k_norm_prep could not stage go the general way (norm_entry).
__global__ void __launch_bounds__(256) k_norm_entries_bits(DevBatch b, DevParams p, const hm_chunk* chunks, uint32_t n_chunks,
                                                           const uint64_t* pair_off, uint64_t n_pairs, const uint8_t* pair_flag,
                                                           const unsigned long long* keys, const uint32_t* koff, uint64_t s0, uint64_t nb,
                                                           const uint32_t* site_lo, const uint32_t* site_n, uint32_t* entries,
                                                           uint64_t stride, const uint32_t* cw_off, const uint32_t* calw,
                                                           const uint8_t* cal_ok, const uint32_t* sdiff, const uint32_t* ref2,
                                                           const uint16_t* mask16, uint32_t modal, uint32_t n_slots) {
  __shared__ uint32_t s_w[8][HM_BYREAD_MAX_OPS], s_t[8][HM_BYREAD_MAX_OPS], s_q[8][HM_BYREAD_MAX_OPS];
  const uint64_t pr = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (pr >= n_pairs) return;
  const uint32_t pf = pair_flag[pr];
  if (!(pf & HM_PF_FETCHED)) return;
  const uint32_t c = upper_bound_dev(pair_off, n_chunks + 1, pr) - 1;
  const hm_chunk ch = chunks[c];
  const uint32_t r = ch.read_lo + (uint32_t)(pr - pair_off[c]);
  const int32_t ts = __ldg(b.tstart + r), te = __ldg(b.tend + r);
  const uint32_t n = __ldg(b.n_ops + r);
  if (n == 0) return;
  const uint32_t k_lo = max(koff[c], (uint32_t)s0), k_hi = min(koff[c + 1], (uint32_t)(s0 + nb));
  if (k_lo >= k_hi) return;
  const unsigned long long base = (unsigned long long)c << 36;
  const uint32_t s_lo = warp_lower_bound_u64(keys, k_lo, k_hi, base | ((unsigned long long)(uint32_t)(ts + 1) << 4), lane);
  const uint32_t s_hi = warp_lower_bound_u64(keys, s_lo, k_hi, base | ((unsigned long long)(uint32_t)(te + 2) << 4), lane);
  if (s_lo >= s_hi) return;
  const uint64_t o0 = __ldg(b.op_off + r);
  const bool staged = n <= HM_BYREAD_MAX_OPS && __ldg(cal_ok + r) != 0;
  if (staged) {
    for (uint32_t k = lane; k < n; k += 32) {
      s_w[wid][k] = __ldg(b.ops + o0 + k); s_t[wid][k] = __ldg(b.op_t + o0 + k); s_q[wid][k] = __ldg(b.op_q + o0 + k);
    }
    __syncwarp();
  }
  const uint64_t bq0 = __ldg(b.bq_off + r), sq0 = __ldg(b.seq_off + r);
  const uint32_t* cw = calw + __ldg(cw_off + r);
  const uint32_t w_first = (uint32_t)ts >> 5;
  for (uint32_t ki = s_lo + lane; ki < s_hi; ki += 32) {
    const uint32_t li = ki - (uint32_t)s0;
    const uint32_t slot = r - __ldg(site_lo + li);
    if (slot >= n_slots || slot >= __ldg(site_n + li)) continue; // pileups deeper than the slots: k_norm_reduce computes these itself
    const int32_t pos = (int32_t)((__ldg(keys + ki) >> 4) & 0xffffffffull) - 1;
    uint32_t e;
    if (!staged) e = norm_entry(b, p, ch, pf, r, pos);
    else {
      const uint32_t off = (uint32_t)(pos - ts);
      uint32_t lo = 0, hi = n; // last op with op_t <= off
      while (lo < hi) { const uint32_t m = (lo + hi) >> 1; if (s_t[wid][m] <= off) lo = m + 1; else hi = m; }
      const int k = (int)lo - 1;
      int ins = 0;
      for (int j = k; j >= 0 && s_t[wid][j] == off; j--) ins += ((s_w[wid][j] & 3u) == HM_OP_INS);
      const uint32_t wd = s_w[wid][k], kind = wd & 3u, t_op = s_t[wid][k], q0 = s_q[wid][k];
      const uint32_t rl = (uint32_t)op_ref_len(wd);
      uint32_t a = HM_ENT_NONE, bq = 0, cnt = 0;
      if (rl != 0 && off < t_op + rl) {
        if (kind == HM_OP_DEL) a = 5u;
        else {
          const uint32_t q = q0 + (kind == HM_OP_MATCH ? off - t_op : 0u);
          bool is_modal = false;
          if (mask16 != nullptr) { const uint64_t bit = bq0 + q; is_modal = (__ldg(mask16 + (bit >> 4)) >> (bit & 15u)) & 1u; }
          bq = is_modal ? modal : (uint32_t)b.bq[bq0 + q];
          if (kind == HM_OP_SUB) { a = (wd >> 5) & 3u; cnt = (pf & HM_PF_PASS) ? 1u : 0u; } // normcounts.py:95-108: always counted
          else {
            const bool differs = (__ldg(sdiff + ((uint32_t)pos >> 5)) >> ((uint32_t)pos & 31u)) & 1u;
            a = differs ? (uint32_t)((b.seq[sq0 + (q >> 2)] >> (2 * (q & 3u))) & 3u)
                        : ((__ldg(ref2 + ((uint32_t)pos >> 4)) >> (2u * ((uint32_t)pos & 15u))) & 3u);
            if (pf & HM_PF_PASS) cnt = (__ldg(cw + (((uint32_t)pos >> 5) - w_first)) >> ((uint32_t)pos & 31u)) & 1u;
          }
        }
      }
      e = a | (bq << 3) | ((uint32_t)min(ins, 255) << 11) | (((pf >> HM_PF_HAP_SHIFT) & 3u) << 19) | (cnt << 21);
    }
    entries[(uint64_t)slot * stride + li] = e;
  }
}

// ============================================================================ k_norm_bits
// carry-save adder: (h, l) = a + b + c per bit
#define NB_CSA(h, l, a, b, c) do { const uint32_t u_ = (a) ^ (b); (h) = ((a) & (b)) | (u_ & (c)); (l) = u_ ^ (c); } while (0)

// eight one-bit-per-position words added into the bit-sliced counter P (P[k] = bit k of the 32 counts): 7 carry-save
// adders and one ripple of the weight-8 word
__device__ __forceinline__ void bits_add8(uint32_t (&P)[8], const uint32_t (&x)[8]) {
  uint32_t tA, tB, fA, fB, e;
  NB_CSA(tA, P[0], P[0], x[0], x[1]);
  NB_CSA(tB, P[0], P[0], x[2], x[3]);
  NB_CSA(fA, P[1], P[1], tA, tB);
  NB_CSA(tA, P[0], P[0], x[4], x[5]);
  NB_CSA(tB, P[0], P[0], x[6], x[7]);
  NB_CSA(fB, P[1], P[1], tA, tB);
  NB_CSA(e, P[2], P[2], fA, fB);
#pragma unroll
  for (int k = 3; k < 8; k++) { const uint32_t t = P[k] & e; P[k] ^= e; e = t; }
}
// positions whose count is >= k
__device__ __forceinline__ uint32_t bits_ge(const uint32_t (&P)[8], int k) {
  if (k <= 0) return 0xffffffffu;
  if (k > 255) return 0u;
  uint32_t gt = 0u, eq = 0xffffffffu;
#pragma unroll
  for (int bq = 7; bq >= 0; bq--) {
    const uint32_t kb = ((k >> bq) & 1) ? 0xffffffffu : 0u;
    gt |= eq & P[bq] & ~kb;
    eq &= ~(P[bq] ^ kb);
  }
  return gt | eq;
}
// sum of the counts over the positions of mask m
__device__ __forceinline__ uint32_t bits_sum(const uint32_t (&P)[8], uint32_t m) {
  uint32_t s = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) s += (uint32_t)__popc(P[k] & m) << k;
  return s;
}

// per span of k_norm_bits: chunk, origin on the 1024 grid, the file-order range of reads that can cover one of its
// positions (running-max(tend) > first position, tstart < end) — so the warps of k_norm_bits do not search
__global__ void __launch_bounds__(256) k_span_ranges(DevBatch b, const hm_chunk* chunks, uint32_t n_chunks, const uint64_t* span_off,
                                                     uint64_t n_spans, uint4* span_info) {
  const uint64_t span = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (span >= n_spans) return;
  const uint32_t c = upper_bound_dev(span_off, n_chunks + 1, span) - 1;
  const hm_chunk ch = chunks[c];
  const int32_t s0 = (int32_t)(((uint32_t)(ch.start >> 10) + (uint32_t)(span - __ldg(span_off + c))) << 10);
  const int32_t lo_pos = max(s0, ch.start), hi_pos = min(s0 + NB_SPAN, ch.end);
  const uint32_t n_in = ch.read_hi - ch.read_lo;
  const uint32_t r_lo = ch.read_lo + count_le_kary_i32(b.pmax_tend + ch.read_lo, n_in, lo_pos);
  const uint32_t r_hi = ch.read_lo + count_le_kary_i32(b.tstart + ch.read_lo, n_in, hi_pos - 1);
  span_info[span] = make_uint4(c, (uint32_t)s0, r_lo, r_hi);
}

// thr[n]: the smallest callable count that certifies a pure position of depth n (host, make_norm_cert), 0xffff: none.
// md_k: depth >= md_k is "read_depth > md_threshold" (256: never).
template <bool kPhase>
__global__ void __launch_bounds__(32 * NB_BITS_WARPS, kPhase ? 4 : 6) k_norm_bits(DevBatch b, DevParams p, const uint16_t* thr, int n_min, int md_k, const hm_chunk* chunks,
                                                                   uint32_t n_chunks, const uint64_t* pair_off, const uint8_t* pair_flag,
                                                                   const uint4* span_info, uint64_t n_spans, const uint32_t* cw_off,
                                                                   const uint32_t* calw, const uint32_t* impure, const uint8_t* tri8,
                                                                   NormOut* out, uint32_t* push_words, uint32_t* span_cnt) {
  __shared__ unsigned long long s_ccs[HM_TRI_BINS], s_ref[HM_TRI_BINS], s_log[HM_NORM_LOG_LEN];
  __shared__ unsigned int s_wccs[NB_BITS_WARPS][HM_TRI_BINS + 1], s_wref[NB_BITS_WARPS][HM_TRI_BINS + 1];
  __shared__ uint16_t s_thr[256];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  for (int i = tid; i < NB_BITS_WARPS * (HM_TRI_BINS + 1); i += blockDim.x) { (&s_wccs[0][0])[i] = 0; (&s_wref[0][0])[i] = 0; }
  if (tid < HM_TRI_BINS) { s_ccs[tid] = 0; s_ref[tid] = 0; }
  if (tid < HM_NORM_LOG_LEN) s_log[tid] = 0;
  for (int i = tid; i < 256; i += blockDim.x) s_thr[i] = thr[i];
  __syncthreads();

  for (uint64_t span = (uint64_t)blockIdx.x * NB_BITS_WARPS + wid; span < n_spans; span += (uint64_t)gridDim.x * NB_BITS_WARPS) {
    const uint4 si = __ldg(span_info + span); // chunk, origin, read range (k_span_ranges)
    const uint32_t c = si.x, r_lo = si.z, r_hi = si.w;
    const hm_chunk ch = chunks[c];
    const int32_t s0 = (int32_t)si.y;
    const int32_t lo_pos = max(s0, ch.start), hi_pos = min(s0 + NB_SPAN, ch.end);
    const bool deep = r_hi > r_lo && r_hi - r_lo > 255u; // the 8-bit counters would overflow: every position to the exact pass
    const uint64_t pbase = __ldg(pair_off + c);
    const int32_t P0 = s0 + 32 * lane;
    const uint32_t W = (uint32_t)P0 >> 5;
    uint32_t N[8] = {0, 0, 0, 0, 0, 0, 0, 0}, C[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    uint32_t H0[8] = {0, 0, 0, 0, 0, 0, 0, 0}, H1[8] = {0, 0, 0, 0, 0, 0, 0, 0}; // kPhase only
    uint32_t n_touch = 0; // reads that cover at least one of this lane's positions: an upper bound of every depth here
    if (!deep) {
      for (uint32_t base = r_lo; base < r_hi; base += 32) {
        const uint32_t rr = base + (uint32_t)lane;
        int32_t l_ts = 0, l_te = 0;
        uint32_t l_off = 0, l_pf = 0;
        if (rr < r_hi) {
          l_pf = pair_flag[pbase + (rr - ch.read_lo)];
          l_ts = __ldg(b.tstart + rr); l_te = __ldg(b.tend + rr);
          l_off = __ldg(cw_off + rr);
          if (!(l_pf & HM_PF_FETCHED)) l_te = l_ts; // covers nothing
        }
        const uint32_t cnt = min(32u, r_hi - base);
        for (uint32_t i0 = 0; i0 < cnt; i0 += 8) {
          uint32_t xm[8], xc[8], x0[8], x1[8]; // x0 / x1: kPhase only
#pragma unroll
          for (uint32_t u = 0; u < 8; u++) {
            const int32_t ts = __shfl_sync(HM_FULL, l_ts, (int)(i0 + u)), te = __shfl_sync(HM_FULL, l_te, (int)(i0 + u));
            const uint32_t off = __shfl_sync(HM_FULL, l_off, (int)(i0 + u)), pf = __shfl_sync(HM_FULL, l_pf, (int)(i0 + u));
            const uint32_t m = low_mask(te - P0) & ~low_mask(ts - P0); // lanes past cnt hold ts = te = 0: nothing
            uint32_t cw = 0;
            if (m && (pf & HM_PF_PASS)) cw = __ldg(calw + off + (W - ((uint32_t)ts >> 5))) & m;
            xm[u] = m; xc[u] = cw;
            n_touch += (m != 0u);
            if constexpr (kPhase) {
              const uint32_t hap = (pf >> HM_PF_HAP_SHIFT) & 3u;
              x0[u] = hap == 0u ? m : 0u; x1[u] = hap == 1u ? m : 0u;
            }
          }
          bits_add8(N, xm);
          bits_add8(C, xc);
          if constexpr (kPhase) { bits_add8(H0, x0); bits_add8(H1, x1); }
        }
      }
    }

    // ---- per position, bit-parallel (normcounts.py:317-400)
    const uint4 ta = __ldg(reinterpret_cast<const uint4*>(tri8 + P0)), tb = __ldg(reinterpret_cast<const uint4*>(tri8 + P0) + 1);
    const uint32_t imp = __ldg(impure + W);
    const uint32_t tw[8] = {ta.x, ta.y, ta.z, ta.w, tb.x, tb.y, tb.z, tb.w};
    uint32_t alive = 0;
#pragma unroll
    for (int g = 0; g < 8; g++) { // a byte of 255: not an upper-case A/C/G/T (or past the contig)
      const uint32_t y = ~tw[g];
      const uint32_t nz = ((((y & 0x7f7f7f7fu) + 0x7f7f7f7fu) | y) >> 7) & 0x01010101u;
      alive |= (((nz * 0x00204081u) >> 21) & 15u) << (4 * g);
    }
    alive &= low_mask(hi_pos - P0) & ~low_mask(lo_pos - P0);
    uint32_t push = deep ? alive : (alive & imp);
    uint32_t ok = 0;
    if (!deep) {
      const uint32_t calpos = C[0] | C[1] | C[2] | C[3] | C[4] | C[5] | C[6] | C[7];
      uint32_t rest = alive & ~imp & calpos; // tri_sum != 0 at a pure position
      unsigned t1 = 0, t2 = 0, t8 = 0, t9 = 0;
      if constexpr (kPhase) {
        const uint32_t unph = rest & ~(bits_ge(H0, p.min_hap_count) & bits_ge(H1, p.min_hap_count));
        const unsigned v = bits_sum(C, unph);
        t1 += v; t2 += v;
        rest &= ~unph;
      }
      const uint32_t cert = rest & bits_ge(N, n_min) & bits_ge(C, (int)s_thr[min(n_touch, 255u)]);
      push |= rest & ~cert;
      const uint32_t md = cert & bits_ge(N, md_k);
      const uint32_t low = cert & ~md & ~bits_ge(N, p.min_ref_count);
      ok = cert & ~md & ~low;
      const unsigned v_cert = bits_sum(C, cert);
      t1 += v_cert;
      t8 = bits_sum(C, md);
      t9 = bits_sum(C, low);
      const unsigned t13 = v_cert - t8 - t9;
      unsigned v;
      v = __reduce_add_sync(HM_FULL, t1); if (lane == 0 && v) atomicAdd(&s_log[1], (unsigned long long)v);
      v = __reduce_add_sync(HM_FULL, t2); if (lane == 0 && v) atomicAdd(&s_log[2], (unsigned long long)v);
      v = __reduce_add_sync(HM_FULL, v_cert); if (lane == 0 && v) atomicAdd(&s_log[6], (unsigned long long)v);
      v = __reduce_add_sync(HM_FULL, t8); if (lane == 0 && v) atomicAdd(&s_log[8], (unsigned long long)v);
      v = __reduce_add_sync(HM_FULL, t9); if (lane == 0 && v) atomicAdd(&s_log[9], (unsigned long long)v);
      v = __reduce_add_sync(HM_FULL, t13); if (lane == 0 && v) atomicAdd(&s_log[13], (unsigned long long)v);
    }
    // the 33-bin tallies of the counted positions: the callable counts transposed out of the bit planes, four at a time
    if (__any_sync(HM_FULL, ok != 0u)) {
#pragma unroll
      for (int g = 0; g < 8; g++) {
        const uint32_t o4 = (ok >> (4 * g)) & 15u;
        if (!o4) continue;
        uint32_t cw = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) cw += spread4((C[k] >> (4 * g)) & 15u) << k;
#pragma unroll
        for (int k = 0; k < 4; k++) {
          if (!((o4 >> k) & 1u)) continue;
          const uint32_t tri = (tw[g] >> (8 * k)) & 255u;
          atomicAdd(&s_wref[wid][tri], 1u);
          atomicAdd(&s_wccs[wid][tri], (cw >> (8 * k)) & 255u);
        }
      }
    }
    // the site list of the exact pass: the lane's word and the span's count now, the keys in position order once the
    // counts are scanned (k_span_scan, k_emit_sites) — the list comes out sorted, nothing sorts it
    push_words[span * 32 + (uint64_t)lane] = push;
    {
      const uint32_t total = __reduce_add_sync(HM_FULL, (uint32_t)__popc(push));
      if (lane == 0) span_cnt[span] = total;
    }
    // the warp's 32-bit bins into the CTA's 64-bit ones before they can overflow
    __syncwarp();
    for (int i = lane; i < HM_TRI_BINS; i += 32) {
      if (s_wccs[wid][i] > 0x40000000u) {
        atomicAdd(&s_ccs[i], (unsigned long long)atomicExch(&s_wccs[wid][i], 0u));
        atomicAdd(&s_ref[i], (unsigned long long)atomicExch(&s_wref[wid][i], 0u));
      }
    }
    __syncwarp();
  }
  __syncwarp();
  for (int i = lane; i < HM_TRI_BINS; i += 32) {
    if (s_wccs[wid][i]) atomicAdd(&s_ccs[i], (unsigned long long)s_wccs[wid][i]);
    if (s_wref[wid][i]) atomicAdd(&s_ref[i], (unsigned long long)s_wref[wid][i]);
  }
  __syncthreads();
  if (tid < HM_TRI_BINS) {
    if (s_ccs[tid]) atomicAdd(&out->ccs_tri[tid], s_ccs[tid]);
    if (s_ref[tid]) atomicAdd(&out->ref_tri[tid], s_ref[tid]);
  }
  if (tid < HM_NORM_LOG_LEN && s_log[tid]) atomicAdd(&out->log[tid], s_log[tid]);
}

// exclusive scan of the spans' site counts -> span_dst[0 .. n_spans], *n_sites = their sum (one CTA: every thread owns a
// run of consecutive spans, one block scan of the run totals)
__global__ void __launch_bounds__(1024) k_span_scan(const uint32_t* span_cnt, uint64_t n_spans, uint32_t* span_dst, unsigned long long* n_sites) {
  __shared__ uint32_t s_warp[33];
  const uint64_t per = (n_spans + blockDim.x - 1) / blockDim.x;
  const uint64_t i0 = min((uint64_t)threadIdx.x * per, n_spans), i1 = min(i0 + per, n_spans);
  uint32_t local = 0;
  for (uint64_t i = i0; i < i1; i++) local += span_cnt[i];
  uint32_t total;
  uint32_t run = block_excl_scan(local, s_warp, &total);
  for (uint64_t i = i0; i < i1; i++) { const uint32_t v = span_cnt[i]; span_dst[i] = run; run += v; }
  if (threadIdx.x == 0) { span_dst[n_spans] = total; *n_sites = (unsigned long long)total; }
}

// the keys (chunk << 36 | (position + 1) << 4) of the listed positions, span by span and ascending inside a span: sorted
__global__ void __launch_bounds__(256) k_emit_sites(const uint4* span_info, uint64_t n_spans, const uint32_t* push_words, const uint32_t* span_dst,
                                                    unsigned long long* sites) {
  const uint64_t span = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (span >= n_spans) return;
  const uint32_t d0 = __ldg(span_dst + span);
  if (__ldg(span_dst + span + 1) == d0) return;
  const uint4 si = __ldg(span_info + span);
  uint32_t todo = __ldg(push_words + span * 32 + (uint64_t)lane);
  const uint32_t np = (uint32_t)__popc(todo);
  uint32_t incl = np;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(HM_FULL, incl, d); if (lane >= d) incl += t; }
  unsigned long long at = (unsigned long long)d0 + (incl - np);
  const int32_t P0 = (int32_t)si.y + 32 * lane;
  while (todo) {
    const int bit = __ffs(todo) - 1;
    todo &= todo - 1;
    sites[at++] = ((unsigned long long)si.x << 36) | ((unsigned long long)(uint32_t)(P0 + bit + 1) << 4);
  }
}
