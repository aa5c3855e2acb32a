// kernels.cuh — sm_100a device code of the himut per-region calling path (`himut call`).
//
//   k_read_scan     cs op stream -> per-op reference / query prefix positions, mismatch list,
//                   match / sub / indel totals, whole-read BQ sum, read gates
//                   (cslib.cs2tuple + cs2subindel, src/himut/cslib.py:13-64;
//                    bamlib.get_qv / get_blast_sequence_identity, src/himut/bamlib.py:34-63;
//                    read gates of caller.py:310-317)
//   k_candidates    per (chunk, read) pair: fetch rule, [--phase: read haplotype], gates,
//                   then trim + mismatch-window filter of every substitution
//                   (bamlib.get_tsbs_candidates, src/himut/bamlib.py:69-86,222-282;
//                    haplib.get_ccs_hap, src/himut/haplib.py:46-83)
//   k_site_range / k_site_entries_by_read / k_site_reduce
//                   per distinct candidate: the pileup column of the chunk's reads at the site
//                   (caller.update_allelecounts, caller.py:44-72) gathered with one warp per
//                   (chunk, read), then per site in file order: counts, ordered fp64 sums,
//                   10-genotype PL / GQ (gtlib.py:72-174), germline restatement test and the
//                   filter cascade (caller.py:324-621) -> record
//
// All streaming, integer / byte work plus ordered fp64 adds; no tensor-core work exists on
// this path.  fp64 sums use __dadd_rn / __dmul_rn so nothing is contracted into FMAs: the
// reference's Python float adds are plain IEEE operations and GQ = int(PL2 - PL1) is taken
// from them.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/himut_b200.h"

#define HM_FULL 0xffffffffu

struct DevBatch {
  uint64_t n_reads;
  const int32_t* tstart;
  const int32_t* tend;
  const int32_t* qstart;
  const int32_t* qlen;
  const uint8_t* mapq;
  const uint8_t* flags;
  const uint32_t* qname_id;
  const uint64_t* seq_off;
  const uint64_t* bq_off;
  const uint64_t* op_off;
  const uint32_t* n_ops;
  const uint8_t* seq;
  const uint8_t* bq;
  const uint32_t* ops;
  // derived by k_read_scan
  uint32_t* op_t;  // reference offset (from tstart) at the start of each op
  uint32_t* op_q;  // query position at the start of each op
  int32_t* mm_pos; // per read, at op_off: 1-based positions of cs2subindel's mismatch_lst
  unsigned long long* bq_total;
  int32_t* n_match;
  int32_t* n_sub;
  int32_t* ins_len;
  int32_t* del_len;
  int32_t* n_mm;
  uint8_t* gate;            // 1: passes the qv / mapq / identity / qlen gates
  const int32_t* pmax_tend; // running maximum of tend (host computed)
};

// scalar worker arguments, by value
struct DevParams {
  int32_t min_qv, min_mapq, qlen_lower_limit, qlen_upper_limit, min_gq, min_bq;
  int32_t max_mismatch_count, mismatch_window, min_ref_count, min_alt_count, min_hap_count;
  int32_t phase, non_human_sample, create_panel_of_normals;
  double min_sequence_identity, min_trim, md_threshold;
};

// per-BQ genotype terms and priors (hm_params.lut_*, log10_prior)
struct DevTables {
  double lut[3][256]; // 0 hom, 1 het, 2 err
  double log10_prior[4];
};
__constant__ DevTables c_tab;

struct DevPhase {
  const int32_t* hpos;
  const uint8_t* href;
  const uint8_t* halt;
  const uint8_t* hbit;
  const uint64_t* set_off;
  uint32_t n_sets;
};

// the three per-BQ tables again, in global memory: lanes index them with different bq, which
// would serialise on the constant cache
struct DevLut { const double* lut; }; // [3][256]

struct DevSets {
  const uint64_t* common;
  uint64_t n_common;
  const uint64_t* pon;
  uint64_t n_pon;
};

// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg_stream16(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p));
  return v;
}
__device__ __forceinline__ uint32_t sum4(uint32_t w, uint32_t acc) { return __dp4a(w, 0x01010101u, acc); }

__device__ __forceinline__ int op_ref_len(uint32_t w) {
  uint32_t kind = w & 3u, v = w >> 2;
  return kind == HM_OP_MATCH ? (int)v : kind == HM_OP_SUB ? 1 : kind == HM_OP_DEL ? (int)v : 0;
}
__device__ __forceinline__ int op_qry_len(uint32_t w) {
  uint32_t kind = w & 3u, v = w >> 2;
  return kind == HM_OP_MATCH ? (int)v : kind == HM_OP_SUB ? 1 : kind == HM_OP_INS ? (int)v : 0;
}

// whole-read quality sum of read r for a warp (np.mean(bq_int_lst) is an exact integer sum divided once): the read's
// qualities as 16-byte words, 4 in flight per lane, summed with dp4a; every lane returns the total
__device__ __forceinline__ unsigned long long warp_bq_sum(const DevBatch& b, uint64_t r, int32_t qlen, int lane) {
  const uint8_t* bq = b.bq + b.bq_off[r];
  const uint4* q4 = reinterpret_cast<const uint4*>(bq);
  const int n16 = qlen >> 4;
  uint32_t acc = 0;
  int i = lane;
  for (; i + 96 < n16; i += 128) {
    uint4 a0 = ldg_stream16(q4 + i), a1 = ldg_stream16(q4 + i + 32), a2 = ldg_stream16(q4 + i + 64), a3 = ldg_stream16(q4 + i + 96);
    acc = sum4(a0.x, acc); acc = sum4(a0.y, acc); acc = sum4(a0.z, acc); acc = sum4(a0.w, acc);
    acc = sum4(a1.x, acc); acc = sum4(a1.y, acc); acc = sum4(a1.z, acc); acc = sum4(a1.w, acc);
    acc = sum4(a2.x, acc); acc = sum4(a2.y, acc); acc = sum4(a2.z, acc); acc = sum4(a2.w, acc);
    acc = sum4(a3.x, acc); acc = sum4(a3.y, acc); acc = sum4(a3.z, acc); acc = sum4(a3.w, acc);
  }
  for (; i < n16; i += 32) {
    uint4 a0 = ldg_stream16(q4 + i);
    acc = sum4(a0.x, acc); acc = sum4(a0.y, acc); acc = sum4(a0.z, acc); acc = sum4(a0.w, acc);
  }
  for (int j = (n16 << 4) + lane; j < qlen; j += 32) acc += bq[j];
  unsigned long long tot = acc;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) tot += __shfl_xor_sync(HM_FULL, tot, d);
  return tot;
}

// ============================================================================ k_read_scan
// One warp per read.  Phase 1: 32 ops at a time, warp inclusive scan of (ref_len, qry_len).
// Phase 2: the read's quality sum (warp_bq_sum).
__global__ void __launch_bounds__(256) k_read_scan(DevBatch b, DevParams p) {
  const uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= b.n_reads) return;
  const uint64_t o0 = b.op_off[r];
  const uint32_t nops = b.n_ops[r];
  const int32_t tstart = b.tstart[r];
  const int32_t qlen = b.qlen[r];
  uint32_t t_carry = 0, q_carry = (uint32_t)b.qstart[r];
  int mm_base = 0, nm = 0, ns = 0, il = 0, dl = 0;
  for (uint32_t base = 0; base < nops; base += 32) {
    const uint32_t k = base + lane;
    const bool valid = k < nops;
    const uint32_t w = valid ? __ldg(b.ops + o0 + k) : 0u;
    const uint32_t kind = w & 3u, v = w >> 2;
    const uint32_t rl = (uint32_t)op_ref_len(w), al = (uint32_t)op_qry_len(w);
    uint32_t rs = rl, qs = al;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t a = __shfl_up_sync(HM_FULL, rs, d), c = __shfl_up_sync(HM_FULL, qs, d);
      if (lane >= d) { rs += a; qs += c; }
    }
    const uint32_t t_ex = t_carry + rs - rl, q_ex = q_carry + qs - al;
    if (valid) { b.op_t[o0 + k] = t_ex; b.op_q[o0 + k] = q_ex; }
    const bool is_mm = valid && ((kind == HM_OP_SUB && (v & 7u) != HM_BASE_N) || kind == HM_OP_INS || kind == HM_OP_DEL);
    const uint32_t bal = __ballot_sync(HM_FULL, is_mm);
    if (is_mm) b.mm_pos[o0 + mm_base + __popc(bal & ((1u << lane) - 1u))] = tstart + (int32_t)t_ex + 1;
    mm_base += __popc(bal);
    if (valid) {
      if (kind == HM_OP_MATCH) nm += (int)v;
      else if (kind == HM_OP_SUB) ns += 1;
      else if (kind == HM_OP_INS) il += (int)v;
      else dl += (int)v;
    }
    t_carry += __shfl_sync(HM_FULL, rs, 31);
    q_carry += __shfl_sync(HM_FULL, qs, 31);
  }
  nm = __reduce_add_sync(HM_FULL, nm);
  ns = __reduce_add_sync(HM_FULL, ns);
  il = __reduce_add_sync(HM_FULL, il);
  dl = __reduce_add_sync(HM_FULL, dl);

  const unsigned long long tot = warp_bq_sum(b, r, qlen, lane);

  if (lane == 0) {
    b.bq_total[r] = tot;
    b.n_match[r] = nm; b.n_sub[r] = ns; b.ins_len[r] = il; b.del_len[r] = dl; b.n_mm[r] = mm_base;
    // caller.py:310-317, in order
    bool ok = true;
    const double qv = __ddiv_rn((double)tot, (double)qlen);
    if (qv < (double)p.min_qv) ok = false;
    if ((int)b.mapq[r] < p.min_mapq) ok = false;
    const double ident = __ddiv_rn((double)nm, (double)(nm + ns + il + dl));
    if (ident < p.min_sequence_identity) ok = false;
    if (!(p.qlen_lower_limit < qlen && qlen < p.qlen_upper_limit)) ok = false;
    b.gate[r] = ok ? 1 : 0;
  }
}

// ============================================================================ k_bq_sum
// The resident batch's per-read quality sums (bq_total, the input of the QV gate) when it came with one quality byte
// per base: one warp per read.  A compact upload has k_bq_expand write them instead.
__global__ void __launch_bounds__(256) k_bq_sum(DevBatch b) {
  const uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= b.n_reads) return;
  const unsigned long long tot = warp_bq_sum(b, r, b.qlen[r], lane);
  if (lane == 0) b.bq_total[r] = tot;
}

// ============================================================================ k_bq_expand
// hm_bq_compact -> the one-byte-per-base quality stream.  One warp per read, 16 bases per lane and step: the lane's
// 16 mask bits, a warp scan of the clear-bit counts to find its first exception, then the exceptions dropped into
// the modal-filled 16-byte word.  Bytes past the read's length (padding) are written as 0.  The read's quality sum
// goes to bq_total.
// exc_minmax[2 r], [2 r + 1]: the smallest / largest exception of read r (255 / 0 when it has none): what lets the
// normcounts pass take "BQ >= min_bq" straight from the bitmap (normbits.cuh).
__global__ void __launch_bounds__(256) k_bq_expand(DevBatch b, const uint8_t* mask, const uint8_t* exc, const uint64_t* exc_off,
                                                   uint32_t modal, uint8_t* bq_out, uint8_t* exc_minmax, unsigned long long* bq_total) {
  const uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= b.n_reads) return;
  const uint32_t qlen = (uint32_t)b.qlen[r];
  const uint64_t off = b.bq_off[r];
  const uint16_t* m16 = reinterpret_cast<const uint16_t*>(mask + (off >> 3));
  uint4* out = reinterpret_cast<uint4*>(bq_out + off);
  const uint8_t* ex = exc + exc_off[r];
  const uint32_t n16 = (qlen + 15u) >> 4;
  const uint32_t fill = modal * 0x01010101u;
  uint32_t run = 0; // exceptions consumed by earlier steps
  uint32_t e_min = 255u, e_max = 0u, acc = 0u;
  for (uint32_t base = 0; base < n16; base += 32) {
    const uint32_t i = base + lane;
    uint32_t bits = 0xffffu, valid = 0;
    if (i < n16) {
      bits = __ldg(m16 + i);
      const uint32_t left = qlen - 16u * i;
      valid = left >= 16u ? 0xffffu : ((1u << left) - 1u);
    }
    const uint32_t zeros = ~bits & valid;
    const uint32_t c = __popc(zeros);
    uint32_t incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(HM_FULL, incl, d); if (lane >= d) incl += t; }
    uint32_t at = run + incl - c;
    run += __shfl_sync(HM_FULL, incl, 31);
    if (i < n16) {
      uint32_t o[4];
#pragma unroll
      for (int wd = 0; wd < 4; wd++) {
        const uint32_t v4 = (valid >> (4 * wd)) & 15u;
        uint32_t word = fill & (((v4 * 0x00204081u) & 0x01010101u) * 0xffu); // modal where the base exists, 0 in the padding
        uint32_t z4 = (zeros >> (4 * wd)) & 15u;
        while (z4) {
          const int k = __ffs(z4) - 1;
          z4 &= z4 - 1;
          const uint32_t ev = (uint32_t)__ldg(ex + at);
          e_min = min(e_min, ev); e_max = max(e_max, ev);
          word = (word & ~(0xffu << (8 * k))) | (ev << (8 * k));
          at++;
        }
        o[wd] = word;
        acc = sum4(word, acc);
      }
      out[i] = make_uint4(o[0], o[1], o[2], o[3]);
    }
  }
  e_min = __reduce_min_sync(HM_FULL, e_min);
  e_max = __reduce_max_sync(HM_FULL, e_max);
  unsigned long long tot = acc; // the read's quality sum (bamlib.get_qv divides it once)
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) tot += __shfl_xor_sync(HM_FULL, tot, d);
  if (lane == 0) { exc_minmax[2 * r] = (uint8_t)e_min; exc_minmax[2 * r + 1] = (uint8_t)e_max; bq_total[r] = tot; }
}

// ============================================================================ lookups
// allele of read r at 0-based reference position rpos (tstart <= rpos <= tend):
//   0..3 base, 5 deleted, -1 no base; *bq = quality of the base; *ins = insertions whose
//   reference position is rpos (caller.update_allelecounts: counts[tpos][4] += 1).
//   ref_base: the reference allele at rpos as the caller's site names it.  A batch uploaded without a base
//   stream (hm_read_batch.seq == NULL) takes the bases of its match runs from there: by the meaning of a cs
//   match (cslib.py:22-29) they are the reference's.
__device__ __forceinline__ int read_allele_at(const DevBatch& b, uint64_t r, int32_t rpos, int ref_base, int* bq, int* ins) {
  const uint32_t n = b.n_ops[r];
  *bq = 0; *ins = 0;
  if (n == 0) return -1;
  const uint64_t o0 = b.op_off[r];
  const uint32_t off = (uint32_t)(rpos - b.tstart[r]);
  uint32_t lo = 0, hi = n;
  while (lo < hi) { // last op with op_t <= off
    uint32_t mid = (lo + hi) >> 1;
    if (__ldg(b.op_t + o0 + mid) <= off) lo = mid + 1; else hi = mid;
  }
  const int k = (int)lo - 1;
  int cnt = 0;
  for (int j = k; j >= 0 && __ldg(b.op_t + o0 + j) == off; j--)
    if ((__ldg(b.ops + o0 + j) & 3u) == HM_OP_INS) cnt++;
  *ins = cnt;
  const uint32_t w = __ldg(b.ops + o0 + k);
  const uint32_t kind = w & 3u, v = w >> 2, t0 = __ldg(b.op_t + o0 + k);
  const uint32_t rl = (uint32_t)op_ref_len(w);
  if (rl == 0 || off >= t0 + rl) return -1;
  if (kind == HM_OP_DEL) return 5;
  const uint32_t q = __ldg(b.op_q + o0 + k) + (kind == HM_OP_MATCH ? off - t0 : 0u);
  *bq = b.bq[b.bq_off[r] + q];
  if (kind == HM_OP_SUB) return (int)((v >> 3) & 7u);
  if (!b.seq) return ref_base;
  return (b.seq[b.seq_off[r] + (q >> 2)] >> (2 * (q & 3u))) & 3;
}

template <typename T>
__device__ __forceinline__ uint32_t upper_bound_dev(const T* a, uint32_t n, T x) { // first a[i] > x
  uint32_t lo = 0, hi = n;
  while (lo < hi) { uint32_t m = (lo + hi) >> 1; if (x < __ldg(a + m)) hi = m; else lo = m + 1; }
  return lo;
}
template <typename T>
__device__ __forceinline__ uint32_t lower_bound_dev(const T* a, uint32_t n, T x) { // first a[i] >= x
  uint32_t lo = 0, hi = n;
  while (lo < hi) { uint32_t m = (lo + hi) >> 1; if (__ldg(a + m) < x) lo = m + 1; else hi = m; }
  return lo;
}
__device__ __forceinline__ bool key_in_dev(const uint64_t* a, uint64_t n, uint64_t key) {
  uint64_t lo = 0, hi = n;
  while (lo < hi) { uint64_t m = (lo + hi) >> 1; if (__ldg(a + m) < key) lo = m + 1; else hi = m; }
  return lo < n && __ldg(a + lo) == key;
}

// the match-run base a batch without a base stream takes at a phased hetSNP (hm_set_phase_sets): href 0..3 is the
// reference base itself; 16 + c says "REF has several bases (never equal to a read base), its first base is c"
__device__ __forceinline__ int href_match_base(int hr) { return hr < 4 ? hr : ((hr & 0xf0) == 0x10 ? (hr & 3) : 4); }

// haplib.get_ccs_hap (haplib.py:61-83) for a whole warp: 0 / 1 / 2 (".")
__device__ __forceinline__ int warp_read_hap(const DevBatch& b, uint64_t r, const DevPhase& ph, int set, int lane) {
  if (set < 0 || (uint32_t)set >= ph.n_sets) return 2;
  const uint64_t s0 = ph.set_off[set];
  const uint32_t n = (uint32_t)(ph.set_off[set + 1] - s0);
  const int32_t* hp = ph.hpos + s0;
  const uint32_t idx = upper_bound_dev(hp, n, b.tstart[r]);
  const uint32_t jdx = upper_bound_dev(hp, n, b.tend[r]);
  if (jdx - idx < 2) return 2;
  bool h0 = true, h1 = true;
  for (uint32_t k = idx + lane; k < jdx; k += 32) {
    int bq, ins;
    const int a = read_allele_at(b, r, hp[k] - 1, href_match_base((int)ph.href[s0 + k]), &bq, &ins);
    int bit = 2;
    if (a >= 0 && a < 4) {
      if (a == (int)ph.href[s0 + k]) bit = 0;
      else if (a == (int)ph.halt[s0 + k]) bit = 1;
    }
    const int hb = ph.hbit[s0 + k];
    if (bit != hb) h0 = false;
    if (bit != 1 - hb) h1 = false;
  }
  h0 = __all_sync(HM_FULL, h0);
  h1 = __all_sync(HM_FULL, h1);
  return h0 ? 0 : (h1 ? 1 : 2);
}

// haplib.get_ccs_hap for one thread: the read's ops walked once, merged with the phase set's hetSNPs in position
// order.  Needs nothing k_read_scan derives (no op prefix arrays).  Used where a record has no (chunk, read) pair of
// its own: the records the reference re-fetches at a phase-checked site (caller.py:558) that share a query name with
// a read of the site's pileup.
__device__ __noinline__ int thread_read_hap_walk(const DevBatch& b, uint64_t r, const DevPhase& ph, int set) {
  if (set < 0 || (uint32_t)set >= ph.n_sets) return 2;
  const uint64_t s0 = ph.set_off[set];
  const uint32_t n = (uint32_t)(ph.set_off[set + 1] - s0);
  const int32_t* hp = ph.hpos + s0;
  const int32_t ts = b.tstart[r];
  const uint32_t idx = upper_bound_dev(hp, n, ts);
  const uint32_t jdx = upper_bound_dev(hp, n, b.tend[r]);
  if (jdx - idx < 2) return 2;
  const uint64_t o0 = b.op_off[r];
  const uint32_t nops = b.n_ops[r];
  uint32_t k = 0, t0 = 0, q0 = (uint32_t)b.qstart[r];
  bool h0 = true, h1 = true;
  for (uint32_t i = idx; i < jdx; i++) {
    const uint32_t off = (uint32_t)(hp[i] - 1 - ts);
    int a = -1;
    while (k < nops) { // the op that holds reference offset `off`
      const uint32_t w = __ldg(b.ops + o0 + k);
      const uint32_t rl = (uint32_t)op_ref_len(w);
      if (rl && off < t0 + rl) {
        const uint32_t kind = w & 3u, v = w >> 2;
        if (kind == HM_OP_DEL) a = 5;
        else if (kind == HM_OP_SUB) a = (int)((v >> 3) & 7u);
        else if (!b.seq) a = href_match_base((int)ph.href[s0 + i]);
        else { const uint32_t q = q0 + (off - t0); a = (b.seq[b.seq_off[r] + (q >> 2)] >> (2 * (q & 3u))) & 3; }
        break;
      }
      t0 += rl; q0 += (uint32_t)op_qry_len(w); k++;
    }
    int bit = 2;
    if (a >= 0 && a < 4) {
      if (a == (int)ph.href[s0 + i]) bit = 0;
      else if (a == (int)ph.halt[s0 + i]) bit = 1;
    }
    const int hb = ph.hbit[s0 + i];
    if (bit != hb) h0 = false;
    if (bit != 1 - hb) h1 = false;
  }
  return h0 ? 0 : (h1 ? 1 : 2);
}

// ============================================================================ k_candidates
// One warp per (chunk, read) pair, pairs enumerated chunk-major over [read_lo, read_hi).
// Emits keys chunk << 36 | tpos << 4 | ref << 2 | alt for every substitution that survives
// get_tsbs_candidates and lies in the chunk (is_chunk, caller.py:325).  som_seen is applied
// later on the host, where the chunk order is sequential.
__global__ void __launch_bounds__(256) k_candidates(DevBatch b, DevParams p, DevPhase ph, const hm_chunk* chunks,
                                                    uint32_t n_chunks, const uint64_t* pair_off, uint64_t n_pairs,
                                                    uint8_t* pair_hap, uint8_t* qname_seen,
                                                    unsigned long long* keys, unsigned long long cap,
                                                    unsigned long long* n_keys, int pos_bits) {
  const uint64_t pr = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (pr >= n_pairs) return;
  uint32_t c = upper_bound_dev(pair_off, n_chunks + 1, pr) - 1;
  const hm_chunk ch = chunks[c];
  const uint64_t r = (uint64_t)ch.read_lo + (pr - pair_off[c]);
  if (pair_hap && lane == 0) pair_hap[pr] = 3; // not fetched
  if (b.flags[r] & HM_READ_SECONDARY) return;
  const int32_t tstart = b.tstart[r], tend = b.tend[r];
  if (!(tstart < ch.end && tend > ch.start)) return;
  if (p.phase) {
    const int hap = warp_read_hap(b, r, ph, ch.phase_set, lane);
    if (lane == 0) pair_hap[pr] = (uint8_t)hap;
    if (hap > 1) return;
  }
  if (!b.gate[r]) return;
  if (lane == 0) qname_seen[b.qname_id[r]] = 1;

  const int32_t qlen = b.qlen[r];
  const double trim_s = floor(__dmul_rn(p.min_trim, (double)qlen));
  const double trim_e = ceil(__dmul_rn(__dsub_rn(1.0, p.min_trim), (double)qlen));
  const uint64_t o0 = b.op_off[r];
  const uint32_t nops = b.n_ops[r];
  const int32_t* mm = b.mm_pos + o0;
  const uint32_t nmm = (uint32_t)b.n_mm[r];
  const int w = p.mismatch_window;
  uint32_t mm_seen = 0; // entries of the mismatch list that belong to ops before this batch
  for (uint32_t base = 0; base < nops; base += 32) {
    const uint32_t k = base + lane;
    bool emit = false;
    unsigned long long key = 0;
    uint32_t op = 0, v = 0;
    bool is_mm = false;
    if (k < nops) {
      op = __ldg(b.ops + o0 + k);
      v = op >> 2;
      const uint32_t kind = op & 3u;
      is_mm = (kind == HM_OP_SUB && (v & 7u) != HM_BASE_N) || kind == HM_OP_INS || kind == HM_OP_DEL; // cs2subindel's list
    }
    const uint32_t mbal = __ballot_sync(HM_FULL, is_mm);
    const int rank = (int)(mm_seen + __popc(mbal & ((1u << lane) - 1u))); // this op's own entry in the mismatch list
    mm_seen += __popc(mbal);
    if (k < nops && (op & 3u) == HM_OP_SUB && (v & 7u) != HM_BASE_N) {
      const int32_t tpos = tstart + (int32_t)b.op_t[o0 + k] + 1;
      const int32_t qpos = (int32_t)b.op_q[o0 + k];
      if (ch.start <= tpos && tpos <= ch.end && !((double)qpos < trim_s) && !((double)qpos > trim_e)) {
        // bamlib.get_mismatch_range
        const int qs = qpos - w, qe = qpos + w;
        int u, d;
        if (qs < 0) { u = w + qs; d = w + (-qs); }
        else if (qe > qlen) { u = w + (qe - qlen); d = qlen - qpos; }
        else { u = w; d = w; }
        // mismatches with tpos - u <= x <= tpos + d, minus this one: walk outwards from the op's own entry
        // (bisect_right - bisect_left - 1, bamlib.py:266-282; the list is sorted and mm[rank] == tpos)
        int cnt = 0;
        for (int j = rank + 1; j < (int)nmm && __ldg(mm + j) <= tpos + d; j++) cnt++;
        for (int j = rank - 1; j >= 0 && __ldg(mm + j) >= tpos - u; j--) cnt++;
        if (!(cnt > p.max_mismatch_count)) {
          emit = true;
          // sort key: chunk | position inside the chunk | ref | alt, packed so the radix sort sees as few bits as
          // possible; k_expand_keys turns it into chunk << 36 | tpos << 4 | ref << 2 | alt afterwards
          key = ((unsigned long long)c << (pos_bits + 4)) | ((unsigned long long)(uint32_t)(tpos - ch.start) << 4) | ((v & 3u) << 2) | ((v >> 3) & 3u);
        }
      }
    }
    const uint32_t bal = __ballot_sync(HM_FULL, emit);
    if (bal) {
      unsigned long long at = 0;
      if (lane == 0) at = atomicAdd(n_keys, (unsigned long long)__popc(bal));
      at = __shfl_sync(HM_FULL, at, 0);
      if (emit) {
        const unsigned long long slot = at + __popc(bal & ((1u << lane) - 1u));
        if (slot < cap) keys[slot] = key;
      }
    }
  }
}

// compact sort key -> chunk << 36 | tpos << 4 | ref << 2 | alt (order is preserved: same fields, same significance)
__global__ void k_expand_keys(unsigned long long* keys, const unsigned long long* n_keys_dev, const hm_chunk* chunks, int pos_bits) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= *n_keys_dev) return;
  const unsigned long long k = keys[i];
  const uint32_t c = (uint32_t)(k >> (pos_bits + 4));
  const uint32_t rel = (uint32_t)((k >> 4) & ((1ull << pos_bits) - 1ull));
  keys[i] = ((unsigned long long)c << 36) | ((unsigned long long)(uint32_t)(chunks[c].start + (int32_t)rel) << 4) | (k & 15ull);
}

// ============================================================================ genotype model
// gtlib.gt_lst (gtlib.py:9) as base codes A0 T1 G2 C3
__device__ __constant__ int8_t c_gt_b1[10] = {0, 1, 3, 2, 1, 3, 2, 3, 2, 2};
__device__ __constant__ int8_t c_gt_b2[10] = {0, 0, 0, 0, 1, 1, 1, 3, 3, 2};

__device__ __forceinline__ int gt_state_dev(int b1, int b2, int ref) { // 0 homref 1 het 2 hetalt 3 homalt
  if (b1 == ref && b2 == ref) return 0;
  if ((b1 == ref) != (b2 == ref)) return 1;
  if (b1 != b2) return 2;
  return 3;
}

// PL of genotype g from the 12 ordered sums S[allele][kind] (gtlib.get_log10_gt_pD,
// gtlib.py:72-96): A,T,G,C terms added left to right from 0, then the prior, then * -10.
// skip >= 0 leaves that allele out (get_germ_gq with a 1-char alt, normcounts.py:389).
__device__ __forceinline__ double gt_pl_dev(const double S[4][3], int g, int ref, int skip) {
  const int b1 = c_gt_b1[g], b2 = c_gt_b2[g];
  double acc = 0.0;
#pragma unroll
  for (int base = 0; base < 4; base++) {
    if (base == skip) continue;
    int kind;
    if (b1 == b2 && base == b1) kind = 0;
    else if (b1 != b2 && (base == b1 || base == b2)) kind = 1;
    else kind = 2;
    acc = __dadd_rn(acc, S[base][kind]);
  }
  acc = __dadd_rn(acc, c_tab.log10_prior[gt_state_dev(b1, b2, ref)]);
  return __dmul_rn(-10.0, acc);
}

// gtlib.get_argmin_gt (gtlib.py:113-119)
__device__ __forceinline__ int argmin_gt_dev(const double pl[10], int* gq, bool* tie) {
  int best = 0;
#pragma unroll
  for (int g = 1; g < 10; g++) if (pl[g] < pl[best]) best = g;
  double second = __longlong_as_double(0x7ff0000000000000ll);
#pragma unroll
  for (int g = 0; g < 10; g++) if (g != best && pl[g] < second) second = pl[g];
  const double d = __dsub_rn(second, pl[best]);
  *gq = d < 99.0 ? (int)d : 99;
  *tie = (second == pl[best]);
  return best;
}

// ---- searches with short dependency chains -------------------------------------------------
// number of elements <= x in sorted a[0..n): 8-ary, the 7 pivots of a level are independent loads
__device__ __forceinline__ uint32_t count_le_kary(const uint32_t* a, uint32_t n, uint32_t x) {
  uint32_t lo = 0, len = n;
  while (len > 8) {
    const uint32_t step = (len + 7) >> 3, end = lo + len;
    uint32_t c = 0;
#pragma unroll
    for (uint32_t i = 1; i < 8; i++) {
      const uint32_t idx = lo + step * i - 1;
      if (idx < end) c += (__ldg(a + idx) <= x);
    }
    lo += c * step;
    len = min(step, end - lo);
  }
  uint32_t c = 0;
#pragma unroll
  for (uint32_t i = 0; i < 8; i++)
    if (i < len) c += (__ldg(a + lo + i) <= x);
  return lo + c;
}
__device__ __forceinline__ uint32_t count_le_kary_i32(const int32_t* a, uint32_t n, int32_t x) {
  uint32_t lo = 0, len = n;
  while (len > 8) {
    const uint32_t step = (len + 7) >> 3, end = lo + len;
    uint32_t c = 0;
#pragma unroll
    for (uint32_t i = 1; i < 8; i++) {
      const uint32_t idx = lo + step * i - 1;
      if (idx < end) c += (__ldg(a + idx) <= x);
    }
    lo += c * step;
    len = min(step, end - lo);
  }
  uint32_t c = 0;
#pragma unroll
  for (uint32_t i = 0; i < 8; i++)
    if (i < len) c += (__ldg(a + lo + i) <= x);
  return lo + c;
}
// warp-cooperative: number of elements of sorted a[0..n) that are < x (strict) or <= x
template <bool kStrict>
__device__ __forceinline__ uint32_t warp_count_below(const int32_t* a, uint32_t n, int32_t x, int lane) {
  uint32_t lo = 0, len = n;
  while (len > 32) {
    const uint32_t step = (len + 32) / 33, end = lo + len;
    const uint32_t idx = lo + step * (lane + 1) - 1;
    bool below = false;
    if (idx < end) { const int32_t v = __ldg(a + idx); below = kStrict ? (v < x) : (v <= x); }
    const uint32_t c = __popc(__ballot_sync(HM_FULL, below));
    lo += c * step;
    len = min(step, end - lo);
  }
  bool below = false;
  if ((uint32_t)lane < len) { const int32_t v = __ldg(a + lo + lane); below = kStrict ? (v < x) : (v <= x); }
  return lo + __popc(__ballot_sync(HM_FULL, below));
}

// read_allele_at with the 8-ary op search
__device__ __forceinline__ int read_allele_fast(const DevBatch& b, uint32_t r, int32_t rpos, int32_t ts, int ref_base, int* bq, int* ins) {
  const uint32_t n = __ldg(b.n_ops + r);
  *bq = 0; *ins = 0;
  if (n == 0) return -1;
  const uint64_t o0 = __ldg(b.op_off + r);
  const uint32_t off = (uint32_t)(rpos - ts);
  const int k = (int)count_le_kary(b.op_t + o0, n, off) - 1;
  int cnt = 0;
  for (int j = k; j >= 0 && __ldg(b.op_t + o0 + j) == off; j--)
    if ((__ldg(b.ops + o0 + j) & 3u) == HM_OP_INS) cnt++;
  *ins = cnt;
  const uint32_t w = __ldg(b.ops + o0 + k);
  const uint32_t kind = w & 3u, v = w >> 2, t0 = __ldg(b.op_t + o0 + k);
  const uint32_t rl = (uint32_t)op_ref_len(w);
  if (rl == 0 || off >= t0 + rl) return -1;
  if (kind == HM_OP_DEL) return 5;
  const uint32_t q = __ldg(b.op_q + o0 + k) + (kind == HM_OP_MATCH ? off - t0 : 0u);
  *bq = b.bq[__ldg(b.bq_off + r) + q];
  if (kind == HM_OP_SUB) return (int)((v >> 3) & 7u);
  if (!b.seq) return ref_base;
  return (b.seq[__ldg(b.seq_off + r) + (q >> 2)] >> (2 * (q & 3u))) & 3;
}

// read_allele_fast without the op prefix arrays (the fused path does not keep them in HBM): one walk over the read's
// ops.  Only the slots past HM_SITE_SLOTS of very deep pileups are answered this way.
__device__ __noinline__ int read_allele_walk(const DevBatch& b, uint32_t r, int32_t rpos, int32_t ts, int ref_base, int* bq, int* ins) {
  const uint32_t n = __ldg(b.n_ops + r);
  *bq = 0; *ins = 0;
  const uint64_t o0 = __ldg(b.op_off + r);
  const uint32_t off = (uint32_t)(rpos - ts);
  uint32_t t = 0, q = (uint32_t)__ldg(b.qstart + r);
  uint32_t lw = 0, lt = 0, lq = 0;
  bool have = false;
  int cnt = 0;
  for (uint32_t k = 0; k < n; k++) { // the last op that starts at or before `off`; insertions that start at it
    const uint32_t w = __ldg(b.ops + o0 + k);
    if (t > off) break;
    if (t == off && (w & 3u) == HM_OP_INS) cnt++;
    lw = w; lt = t; lq = q; have = true;
    t += (uint32_t)op_ref_len(w); q += (uint32_t)op_qry_len(w);
  }
  *ins = cnt;
  if (!have) return -1;
  const uint32_t kind = lw & 3u, v = lw >> 2;
  const uint32_t rl = (uint32_t)op_ref_len(lw);
  if (rl == 0 || off >= lt + rl) return -1;
  if (kind == HM_OP_DEL) return 5;
  const uint32_t qq = lq + (kind == HM_OP_MATCH ? off - lt : 0u);
  *bq = b.bq[__ldg(b.bq_off + r) + qq];
  if (kind == HM_OP_SUB) return (int)((v >> 3) & 7u);
  if (!b.seq) return ref_base;
  return (b.seq[__ldg(b.seq_off + r) + (qq >> 2)] >> (2 * (qq & 3u))) & 3;
}

// ============================================================================ site kernels
// The pileup column of a candidate site is gathered in three steps so every thread has work and
// the order-sensitive part stays sequential per site:
//   k_site_range    1 thread / distinct candidate: the file-order index range [lo, lo + n) of the
//                   chunk's reads that can touch the site (two 8-ary searches);
//   k_site_entries_by_read
//                   1 warp / (chunk, read): allele, BQ, insertion count, haplotype of that read at
//                   each site it covers, packed into one u32 per (site, read slot), stored slot-major
//                   so the next kernel's reads are coalesced;
//   k_site_reduce   1 thread / candidate: walks the slots in file order — 6 counts, BQ sums, the
//                   12 ordered fp64 sums (caller.update_allelecounts appends in fetch order,
//                   caller.py:44-72), haplotype tallies — then 10-genotype PL / GQ
//                   (gtlib.py:72-135), germline restatement (caller.is_germ_gt), the cascade
//                   (caller.py:349-621) and the record; status tallies and the boundary list for
//                   the host's som_seen replay.
#define HM_SITE_SLOTS 64
#define HM_ENT_NONE 7u

// entry: bits 0-2 allele (0-3 base, 5 deleted, 7 none), 3-10 BQ, 11-18 insertions at the site,
//        19-20 haplotype (0, 1, 2 ".", 3 not fetched), 21 read also covers the next position
// walk: the batch's op prefix arrays are not filled (fused path)
__device__ __forceinline__ uint32_t site_entry(const DevBatch& b, const DevParams& p, const hm_chunk& ch, uint32_t c,
                                               const uint64_t* pair_off, const uint8_t* pair_hap, uint32_t r, int32_t rpos,
                                               int ref_base, bool walk = false) {
  uint32_t e = HM_ENT_NONE;
  if (!(__ldg(b.flags + r) & HM_READ_SECONDARY)) {
    const int32_t ts = __ldg(b.tstart + r), te = __ldg(b.tend + r);
    if (ts < ch.end && te > ch.start && ts <= rpos && rpos <= te) {
      int bq, ins;
      const int a = walk ? read_allele_walk(b, r, rpos, ts, ref_base, &bq, &ins) : read_allele_fast(b, r, rpos, ts, ref_base, &bq, &ins);
      const uint32_t hap = p.phase ? pair_hap[pair_off[c] + (r - ch.read_lo)] : 2u;
      e = (a < 0 ? HM_ENT_NONE : (uint32_t)a) | ((uint32_t)bq << 3) | ((uint32_t)min(ins, 255) << 11) | ((hap & 3u) << 19) |
          ((te > rpos + 1) ? (1u << 21) : 0u); // overlaps [tpos, tpos + 1) (caller.py:558)
    }
  }
  return e;
}

__global__ void __launch_bounds__(256) k_site_range(DevBatch b, const hm_chunk* chunks, const unsigned long long* keys,
                                                    const unsigned long long* n_keys_dev, uint32_t* site_lo, uint32_t* site_n) {
  const uint64_t ki = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (ki >= *n_keys_dev) return;
  const unsigned long long key = keys[ki];
  const hm_chunk ch = chunks[(uint32_t)(key >> 36)];
  const int32_t rpos = (int32_t)((key >> 4) & 0xffffffffull) - 1;
  // reads that can touch rpos, inside the chunk's fetch range: running-max(tend) >= rpos
  // (a trailing insertion sits at tend) and tstart <= rpos
  const uint32_t n_in = ch.read_hi - ch.read_lo;
  const uint32_t lo = count_le_kary_i32(b.pmax_tend + ch.read_lo, n_in, rpos - 1);
  const uint32_t hi = count_le_kary_i32(b.tstart + ch.read_lo, n_in, rpos);
  site_lo[ki] = ch.read_lo + lo;
  site_n[ki] = hi > lo ? hi - lo : 0u;
}

// ---- gather by read ------------------------------------------------------------------------------
// Rather than asking, for every (site, read) pair, "which op of this read holds the site" with a search over
// the read's op arrays in global memory, k_site_entries_by_read turns the loop around: one warp per
// (chunk, read) pair stages the read's op arrays in shared memory once and then serves all the chunk's sites
// the read covers (about 60 per 15 kb read), 32 sites at a time; the only scattered global loads left are the
// site's quality byte and its 2-bit base.  Entries nobody writes (reads that do not reach a site) keep the
// 0xffffffff the buffer is initialised with; k_site_reduce skips them.
#define HM_ENT_UNWRITTEN 0xffffffffu
#define HM_BYREAD_MAX_OPS 192

// warp-cooperative: first index in [lo, hi) with a[i] >= x (32 pivots per round)
__device__ __forceinline__ uint32_t warp_lower_bound_u64(const unsigned long long* a, uint32_t lo, uint32_t hi, unsigned long long x, int lane) {
  while (hi - lo > 32) {
    const uint32_t step = (hi - lo + 32) / 33;
    const uint32_t idx = lo + step * (uint32_t)(lane + 1) - 1;
    const bool below = idx < hi && __ldg(a + idx) < x;
    const uint32_t cnt = __popc(__ballot_sync(HM_FULL, below));
    lo += cnt * step;
    hi = min(hi, lo + step);
  }
  const bool below = lo + (uint32_t)lane < hi && __ldg(a + lo + lane) < x;
  return lo + __popc(__ballot_sync(HM_FULL, below));
}

// first key of each chunk in the sorted distinct keys: koff[c] = lower_bound(keys, c << 36), koff[n_chunks] = n_keys
__global__ void k_chunk_key_ranges(const unsigned long long* keys, const unsigned long long* n_keys_dev, uint32_t n_chunks,
                                   uint32_t* koff) {
  const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c > n_chunks) return;
  const uint64_t n = *n_keys_dev;
  const unsigned long long want = (unsigned long long)c << 36;
  uint64_t lo = 0, hi = n;
  while (lo < hi) { const uint64_t m = (lo + hi) >> 1; if (__ldg(keys + m) < want) lo = m + 1; else hi = m; }
  koff[c] = (uint32_t)lo;
}

// kSeq: the batch has a base stream (false: match runs carry the site's reference allele, hm_read_batch.seq == NULL)
template <bool kSeq>
__global__ void __launch_bounds__(256) k_site_entries_by_read(DevBatch b, DevParams p, const hm_chunk* chunks, uint32_t n_chunks,
                                                              const uint64_t* pair_off, uint64_t n_pairs, const uint8_t* pair_hap,
                                                              const unsigned long long* keys, const uint32_t* koff,
                                                              const uint32_t* site_lo, const uint32_t* site_n, uint32_t* entries,
                                                              uint64_t stride) {
  __shared__ uint32_t s_w[8][HM_BYREAD_MAX_OPS], s_t[8][HM_BYREAD_MAX_OPS], s_q[8][HM_BYREAD_MAX_OPS];
  const uint64_t pr = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (pr >= n_pairs) return;
  const uint32_t c = upper_bound_dev(pair_off, n_chunks + 1, pr) - 1;
  const hm_chunk ch = chunks[c];
  const uint32_t r = ch.read_lo + (uint32_t)(pr - pair_off[c]);
  if (__ldg(b.flags + r) & HM_READ_SECONDARY) return;
  const int32_t ts = __ldg(b.tstart + r), te = __ldg(b.tend + r);
  if (!(ts < ch.end && te > ch.start)) return;
  const uint32_t n = __ldg(b.n_ops + r);
  if (n == 0) return;
  // the chunk's sites with rpos in [ts, te], i.e. tpos in [ts + 1, te + 1]
  const uint32_t k_lo = koff[c], k_hi = koff[c + 1];
  if (k_lo == k_hi) return;
  const unsigned long long base = (unsigned long long)c << 36;
  const unsigned long long want_lo = base | ((unsigned long long)(uint32_t)(ts + 1) << 4);
  const unsigned long long want_hi = base | ((unsigned long long)(uint32_t)(te + 2) << 4);
  const uint32_t s_lo = warp_lower_bound_u64(keys, k_lo, k_hi, want_lo, lane);
  const uint32_t s_hi = warp_lower_bound_u64(keys, s_lo, k_hi, want_hi, lane);
  if (s_lo >= s_hi) return;
  const uint64_t o0 = __ldg(b.op_off + r);
  const bool staged = n <= HM_BYREAD_MAX_OPS;
  if (staged) {
    for (uint32_t k = lane; k < n; k += 32) {
      s_w[wid][k] = __ldg(b.ops + o0 + k); s_t[wid][k] = __ldg(b.op_t + o0 + k); s_q[wid][k] = __ldg(b.op_q + o0 + k);
    }
    __syncwarp();
  }
  const uint64_t bq0 = __ldg(b.bq_off + r), sq0 = kSeq ? __ldg(b.seq_off + r) : 0;
  const uint32_t hap = p.phase ? pair_hap[pr] : 2u;
  for (uint32_t ki = s_lo + lane; ki < s_hi; ki += 32) {
    const uint32_t slot = r - __ldg(site_lo + ki);
    if (slot >= HM_SITE_SLOTS || slot >= __ldg(site_n + ki)) continue; // deep pileups: k_site_reduce computes these itself
    const unsigned long long key = __ldg(keys + ki);
    const int32_t rpos = (int32_t)((key >> 4) & 0xffffffffull) - 1;
    const int ref_base = (int)((key >> 2) & 3);
    int a, bq = 0, ins = 0;
    if (staged) {
      const uint32_t off = (uint32_t)(rpos - ts);
      uint32_t lo = 0, hi = n; // last op with op_t <= off
      while (lo < hi) { const uint32_t m = (lo + hi) >> 1; if (s_t[wid][m] <= off) lo = m + 1; else hi = m; }
      const int k = (int)lo - 1;
      for (int j = k; j >= 0 && s_t[wid][j] == off; j--) ins += ((s_w[wid][j] & 3u) == HM_OP_INS);
      const uint32_t wd = s_w[wid][k], kind = wd & 3u, v = wd >> 2, t_op = s_t[wid][k];
      const uint32_t rl = (uint32_t)op_ref_len(wd);
      if (rl == 0 || off >= t_op + rl) a = -1;
      else if (kind == HM_OP_DEL) a = 5;
      else {
        const uint32_t q = s_q[wid][k] + (kind == HM_OP_MATCH ? off - t_op : 0u);
        bq = b.bq[bq0 + q];
        a = kind == HM_OP_SUB ? (int)((v >> 3) & 7u) : !kSeq ? ref_base : (int)((b.seq[sq0 + (q >> 2)] >> (2 * (q & 3u))) & 3u);
      }
    } else {
      a = read_allele_fast(b, r, rpos, ts, ref_base, &bq, &ins);
    }
    entries[(uint64_t)slot * stride + ki] = (a < 0 ? HM_ENT_NONE : (uint32_t)a) | ((uint32_t)bq << 3) | ((uint32_t)min(ins, 255) << 11) |
                                            ((hap & 3u) << 19) | ((te > rpos + 1) ? (1u << 21) : 0u);
  }
}

// ph / dup_names: two primary records of the batch share a query name.  The reference classifies the records it
//   re-fetches at a phase-checked site by *name* (wt_ccs_set / alt_ccs_set, caller.py:556-567); with unique names
//   that is the record's own allele (the entries' haplotype tallies), with shared names the exact walk below.
// compact_out / n_kept / boundary_pos (fused path, else NULL): the records the host wants (not dropped; not a germline
//   restatement when omit != 0) are written to compact_out only — a block reserves its range with one atomic on
//   *n_kept, inside the block the order is the key order — and a boundary record carries its position there
//   (0xffffffff: not kept).  `out` is not written then.
#ifndef HM_REDUCE_MINB
#define HM_REDUCE_MINB 5 // 96 registers; six CTAs (80 registers, a few spills) run the same, four are 12 % slower
#endif
__global__ void __launch_bounds__(128, HM_REDUCE_MINB) k_site_reduce(DevBatch b, DevParams p, DevSets sets, DevLut lut, DevPhase ph, int dup_names,
                                                     const hm_chunk* chunks,
                                                     const uint64_t* pair_off, const uint8_t* pair_hap, const int32_t* prev_max_end,
                                                     const int32_t* next_min_start, const unsigned long long* keys,
                                                     const unsigned long long* n_keys_dev, const uint32_t* site_lo,
                                                     const uint32_t* site_n, const uint32_t* entries, uint64_t stride,
                                                     hm_site_record* out, unsigned long long* status_hist, uint32_t* boundary_idx,
                                                     hm_site_record* boundary_recs, uint32_t boundary_cap,
                                                     unsigned long long* n_boundary, int* err_flag,
                                                     hm_site_record* compact_out,
                                                     unsigned long long* n_kept, uint32_t* boundary_pos, int omit, uint32_t n_slots) {
  __shared__ unsigned int s_hist[16];
  __shared__ unsigned int s_wkeep[4], s_kbase;
  __shared__ double s_lut[3][256];
  for (int i = threadIdx.x; i < 768; i += blockDim.x) s_lut[i >> 8][i & 255] = __ldg(lut.lut + i);
  if (threadIdx.x < 16) s_hist[threadIdx.x] = 0;
  __syncthreads();
  hm_site_record R;
  bool have_rec = false, keep = false, bnd = false;
  const uint64_t ki = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t n_keys = *n_keys_dev;
  const bool fused = compact_out != nullptr; // no op prefix arrays in HBM then
  if (ki < n_keys) {
    const unsigned long long key = keys[ki];
    const uint32_t c = (uint32_t)(key >> 36);
    const int32_t tpos = (int32_t)((key >> 4) & 0xffffffffull);
    const int ref = (int)((key >> 2) & 3), alt = (int)(key & 3);
    const hm_chunk ch = chunks[c];
    const uint32_t n = site_n[ki], lo = site_lo[ki];

    int cnt[6] = {0, 0, 0, 0, 0, 0}, bqs[4] = {0, 0, 0, 0};
    int hi_bq_alt = 0, h0 = 0, h1 = 0, som_mask = 0;
    bool bq_zero = false;
    double SS[4][3];
#pragma unroll
    for (int x = 0; x < 4; x++) { SS[x][0] = 0.0; SS[x][1] = 0.0; SS[x][2] = 0.0; }
    auto acc = [&](uint32_t e) {
      if (e == HM_ENT_UNWRITTEN) return; // a read of the range that does not reach the site
      const uint32_t a = e & 7u;
      cnt[4] += (int)((e >> 11) & 255u);
      if (a == HM_ENT_NONE) return;
      if (a == 5u) { cnt[5]++; return; }
      const int bq = (int)((e >> 3) & 255u);
      const uint32_t hap = (e >> 19) & 3u;
      const bool next_cov = (e >> 21) & 1u;
      if (bq == 0) bq_zero = true;
      const double x0 = s_lut[0][bq], x1 = s_lut[1][bq], x2 = s_lut[2][bq];
#pragma unroll
      for (int x = 0; x < 4; x++) {
        if ((int)a == x) {
          cnt[x]++; bqs[x] += bq;
          SS[x][0] = __dadd_rn(SS[x][0], x0); SS[x][1] = __dadd_rn(SS[x][1], x1); SS[x][2] = __dadd_rn(SS[x][2], x2);
        }
      }
      if ((int)a == alt && bq >= p.min_bq) hi_bq_alt++;
      if (p.phase && next_cov) {
        if ((int)a == ref) { h0 += (hap == 0u); h1 += (hap == 1u); }
        else if ((int)a == alt) { if (hap == 0u) som_mask |= 1; else if (hap == 1u) som_mask |= 2; }
      }
    };
    // slots in file order: the first HM_SITE_SLOTS from the gathered entries (eight independent loads at a time),
    // deeper pileups computed here
    const uint32_t n_slot = min(n, n_slots);
    for (uint32_t s0 = 0; s0 < n_slot; s0 += 8) {
      uint32_t ev[8];
#pragma unroll
      for (int j = 0; j < 8; j++) ev[j] = (s0 + j < n_slot) ? __ldg(entries + (uint64_t)(s0 + j) * stride + ki) : HM_ENT_UNWRITTEN;
#pragma unroll
      for (int j = 0; j < 8; j++) acc(ev[j]);
    }
    for (uint32_t s = n_slots; s < n; s++) acc(site_entry(b, p, ch, c, pair_off, pair_hap, lo + s, tpos - 1, ref, fused));
    if (bq_zero) *err_flag = HM_ERR_BQ_ZERO;

    double pl[10];
#pragma unroll
    for (int g = 0; g < 10; g++) pl[g] = gt_pl_dev(SS, g, ref, -1);
    int gq; bool tie;
    const int best = argmin_gt_dev(pl, &gq, &tie);
    int g0 = c_gt_b1[best], g1 = c_gt_b2[best];
    const int state = gt_state_dev(g0, g1, ref);
    if (g0 != ref && ((g0 == ref) + (g1 == ref)) == 1) { int t = g0; g0 = g1; g1 = t; } // gtlib.py:133-134
    const int ins_count = cnt[4], del_count = cnt[5];
    const int depth = cnt[0] + cnt[1] + cnt[2] + cnt[3] + cnt[5];
    const int ref_count = cnt[ref], alt_count = cnt[alt];

    // caller.is_germ_gt (caller.py:111-147)
    bool germ;
    if (state == 1) germ = (g0 == ref && g1 == alt);
    else if (state == 2) germ = (cnt[0] + cnt[1] + cnt[2] + cnt[3] == cnt[g0] + cnt[g1]) && (alt == g0 || alt == g1);
    else if (state == 3) germ = (ref_count == 0 && g0 == alt && g1 == alt);
    else germ = (alt == g0);

    int status, phase_set = -1;
    if (germ) status = state == 1 ? HM_ST_GERM_HET : state == 2 ? HM_ST_GERM_HETALT : state == 3 ? HM_ST_GERM_HOMALT : HM_ST_GERM_HOMREF;
    else if (state == 1) status = HM_ST_HET_SITE;
    else if (state == 2) status = HM_ST_HETALT_SITE;
    else if (state == 3) status = HM_ST_HOMALT_SITE;
    else if (del_count != 0 || ins_count != 0) status = HM_ST_INDEL_SITE;
    else {
      const uint64_t skey = ((uint64_t)(uint32_t)tpos << 4) | ((uint64_t)ref << 2) | (uint64_t)alt;
      if (gq < p.min_gq) status = HM_ST_LOW_GQ;
      else if (hi_bq_alt == 0) status = HM_ST_LOW_BQ;
      else if (!p.non_human_sample && !p.create_panel_of_normals && key_in_dev(sets.pon, sets.n_pon, skey)) status = HM_ST_PON;
      else if (!p.non_human_sample && key_in_dev(sets.common, sets.n_common, skey)) status = HM_ST_COMSNP;
      else if (!(ref_count >= p.min_ref_count && alt_count >= p.min_alt_count)) status = HM_ST_LOW_DEPTH;
      else if ((double)depth > p.md_threshold) status = HM_ST_HIGH_DEPTH;
      else {
        status = HM_ST_PASS;
        if (p.phase) { // caller.py:552-603
          if (dup_names) {
            // Query names are shared: do what the reference does.  Every primary record of the file that overlaps
            // [tpos, tpos + 1) (alignments.fetch(chrom, tpos, tpos + 1)) is classified by whether its *name* is
            // among the names of the pileup's ref-allele reads, else of its alt-allele reads; its own haplotype counts.
            h0 = 0; h1 = 0; som_mask = 0;
            const uint32_t r_lo = count_le_kary_i32(b.pmax_tend, (uint32_t)b.n_reads, tpos); // first read with running max(tend) > tpos
            for (uint32_t r = r_lo; r < (uint32_t)b.n_reads && __ldg(b.tstart + r) < tpos + 1; r++) {
              if (!(__ldg(b.tend + r) > tpos) || (__ldg(b.flags + r) & HM_READ_SECONDARY)) continue;
              const uint32_t q = __ldg(b.qname_id + r);
              bool in_wt = false, in_alt = false;
              for (uint32_t s = 0; s < n; s++) {
                if (__ldg(b.qname_id + lo + s) != q) continue;
                const uint32_t e = s < n_slots ? __ldg(entries + (uint64_t)s * stride + ki)
                                               : site_entry(b, p, ch, c, pair_off, pair_hap, lo + s, tpos - 1, ref, fused);
                if (e == HM_ENT_UNWRITTEN) continue;
                const int a = (int)(e & 7u);
                if (a == ref) { in_wt = true; break; }
                if (a == alt) in_alt = true;
              }
              if (!in_wt && !in_alt) continue;
              int hap = 3;
              if (r >= ch.read_lo && r < ch.read_hi) hap = pair_hap[pair_off[c] + (r - ch.read_lo)];
              if (hap == 3) hap = thread_read_hap_walk(b, r, ph, ch.phase_set); // not fetched by this chunk
              if (in_wt) { h0 += (hap == 0); h1 += (hap == 1); }
              else if (hap < 2) som_mask |= 1 << hap;
            }
          }
          if (h0 >= p.min_hap_count && h1 >= p.min_hap_count && (som_mask == 1 || som_mask == 2)) phase_set = ch.start;
          else status = HM_ST_UNPHASED;
        }
      }
    }
    R.tpos = tpos; R.ref = (uint8_t)ref; R.alt = (uint8_t)alt; R.status = (uint8_t)status;
    R.flags = tie ? HM_SITE_PL_TIE : 0;
    R.chunk = (int32_t)c; R.gq = gq;
    R.germ_gt[0] = (uint8_t)g0; R.germ_gt[1] = (uint8_t)g1; R.germ_state = (uint8_t)state; R.pad0 = 0;
#pragma unroll
    for (int x = 0; x < 6; x++) R.counts[x] = cnt[x];
#pragma unroll
    for (int x = 0; x < 4; x++) R.bq_sum[x] = bqs[x];
    const bool ph_eval = p.phase && (status == HM_ST_PASS || status == HM_ST_UNPHASED);
    R.hap_count[0] = ph_eval ? h0 : 0; R.hap_count[1] = ph_eval ? h1 : 0;
    R.som_hap_mask = ph_eval ? som_mask : 0;
    R.phase_set = phase_set;
    have_rec = true;
    keep = !(omit && status >= HM_ST_GERM_HET && status <= HM_ST_GERM_HOMREF);
    bnd = tpos <= prev_max_end[c] || tpos >= next_min_start[c];
    atomicAdd(&s_hist[status], 1u);
  }
  uint32_t pos = 0xffffffffu;
  if (compact_out) { // block-stable compaction: ballot rank inside the warp, warp totals, one atomic per block
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t bal = __ballot_sync(HM_FULL, keep);
    if (lane == 0) s_wkeep[wid] = __popc(bal);
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned int tot = s_wkeep[0] + s_wkeep[1] + s_wkeep[2] + s_wkeep[3];
      s_kbase = tot ? (unsigned int)atomicAdd(n_kept, (unsigned long long)tot) : 0u;
    }
    __syncthreads();
    uint32_t before = 0;
    for (int w = 0; w < wid; w++) before += s_wkeep[w];
    if (keep) { pos = s_kbase + before + __popc(bal & ((1u << lane) - 1u)); compact_out[pos] = R; }
  } else if (have_rec) {
    out[ki] = R;
  }
  if (bnd) { // a copy for the host's som_seen replay
    const unsigned long long at = atomicAdd(n_boundary, 1ull);
    if (at < boundary_cap) { boundary_idx[at] = (uint32_t)ki; boundary_recs[at] = R; if (boundary_pos) boundary_pos[at] = pos; }
  }
  __syncthreads();
  if (threadIdx.x < 16 && s_hist[threadIdx.x]) atomicAdd(status_hist + threadIdx.x, (unsigned long long)s_hist[threadIdx.x]);
}

// Small results go to the host through mapped pinned memory (plain stores over PCIe) instead of the copy engine,
// where they would queue behind a previous call's 20 MB record copy.  words of 4 bytes; *n_src_limit (optional)
// bounds how many `item_words`-sized items of src are worth sending.
// The other way round: a call's few KB of chunk geometry come from mapped pinned host memory through plain loads over
// PCIe, not through the copy engine — there a small copy of this context waits behind the other context's 0.46 GB upload
// (measured: the whole device path of every second call started 9 ms late, tools/step_trace.py --mode e2e).
__global__ void __launch_bounds__(256) k_fetch_block(const uint4* mapped_src, uint4* dst, uint32_t n16) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += gridDim.x * blockDim.x) dst[i] = mapped_src[i];
}

__global__ void k_publish(const uint32_t* src, uint32_t* mapped_dst, uint32_t n_words) {
  for (uint32_t i = threadIdx.x; i < n_words; i += blockDim.x) mapped_dst[i] = src[i];
  __threadfence_system();
}
__global__ void k_publish_items(const uint32_t* src, uint32_t* mapped_dst, uint32_t item_words, uint32_t max_items,
                                const unsigned long long* n_items_dev) {
  const unsigned long long n = min((unsigned long long)max_items, *n_items_dev);
  const uint64_t total = n * item_words;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) mapped_dst[i] = src[i];
  __threadfence_system();
}

// ---- records the reference never emits stay on the device (option HM_OPT_OMIT_RESTATEMENTS) ----------------
// A candidate that merely restates the germline genotype is counted and dropped by the reference
// (caller.py:338-345): its record is needed for the counters and the boundary replay only.  keep flags -> exclusive
// scan (cub) -> stable compaction; the host copies the compact array.
__global__ void k_keep_flags(const hm_site_record* rec, const unsigned long long* n_dev, uint32_t* flags) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= *n_dev) return;
  const uint8_t st = rec[i].status;
  flags[i] = (st >= HM_ST_GERM_HET && st <= HM_ST_GERM_HOMREF) ? 0u : 1u;
}
__global__ void k_compact_records(const hm_site_record* rec, const uint32_t* flags, const uint32_t* pos,
                                  const unsigned long long* n_dev, hm_site_record* out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= *n_dev) return;
  if (flags[i]) out[pos[i]] = rec[i];
}
// dst[i] = src[idx[i]] for the first min(cap, *n_items_dev) entries
__global__ void k_gather_u32(const uint32_t* src, const uint32_t* idx, const unsigned long long* n_items_dev, uint32_t cap, uint32_t* dst) {
  const unsigned long long n = min((unsigned long long)cap, *n_items_dev);
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) dst[i] = src[idx[i]];
}

// number of set bytes in flags[0..n)
__global__ void k_count_flags(const uint8_t* flags, uint64_t n, unsigned long long* out) {
  unsigned long long c = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) c += flags[i] != 0;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(HM_FULL, c, d);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}
