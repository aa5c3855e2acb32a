// callfused.cuh — the fused device path of `himut call` (sm_100a).
//
// The reference piles up every aligned base of every read (caller.update_allelecounts, caller.py:44-72) and then looks
// at the pileup only where a read carries a candidate substitution (caller.py:324-336).  The first version of this
// path (kernels.cuh: k_read_scan -> k_candidates -> library sort -> k_site_entries_by_read -> k_site_reduce) streamed
// the whole quality stream on every call to sum it for the QV gate.  Here no call streams it: the QV gate reads the
// per-read quality sum the batch carries since it became resident (DevBatch.bq_total: k_bq_expand or k_bq_sum), and
// the pileup columns take one quality byte per (site, covering read):
//
//   k_call_pairs   (ops only)  one thread per (chunk, read) pair: cs op walk, mismatch list, QV / MAPQ / identity /
//                  length gates, [--phase] read haplotype, then trim + mismatch-window test of every substitution
//                  (bamlib.get_tsbs_candidates, bamlib.py:69-86) -> candidate keys into the chunk's own segment.
//                  A read that passes every gate counts its query name (num_ccs).
//   k_site_sort    one CTA per 2^17-position tile of a chunk: the chunk's keys -> sorted distinct sites without a
//                  comparison sort: position bitmap in shared memory, popcount prefix = rank, 16-bit (ref, alt) mask
//                  per distinct position (set(somatic_tsbs_candidate_lst), caller.py:324).
//   k_tile_scan    exclusive scan of the per-tile site counts (one CTA); k_site_range2: final key array, the
//                  file-order read range of every site, entry slots initialised.
//   k_call_scan    the pileup entries.  One warp per (chunk, read) pair: the sites the read covers, its op prefixes
//                  in shared memory, the allele of every site and one quality byte per site that has a base.
//   k_site_reduce  (kernels.cuh) per site, reads in file order: counts, ordered fp64 sums, PL / GQ, cascade, record.
//   k_compact_sites  records the host wants, stably compacted (no germline restatements when asked, no dropped sites).
//
// No host synchronisation between the kernels: capacities are bounds known on the host (ops per chunk) or a
// high-water estimate with an overflow flag (distinct sites), counts stay on the device.
#pragma once
#include "kernels.cuh"

#ifndef HC_MAX_OPS
#define HC_MAX_OPS 96                  // ops of a read staged per warp; longer lists use the batch's global op_t / op_q
#endif
#define HC_TILE_BITS 17
#define HC_TILE (1u << HC_TILE_BITS)   // positions per sort tile
#define HC_TILE_WORDS (HC_TILE / 32u)
#define HC_CAPD 4096u                  // distinct positions of a tile kept in shared memory (more: global scratch)
#define HC_SORT_THREADS 512
#define HC_KEY_POS_BITS 27             // a chunk may span < 2^27 positions on this path (else the first version runs)

struct OpView { const uint32_t* w; const uint32_t* t; const uint32_t* q; uint32_t n; };

// allele of a read at reference offset `off` from its start: -1 none, 5 deleted, 8 the base of a match run, else the
// substituted base; *q = query position of the base, *ins = insertions whose reference position is `off`
// (same rules as read_allele_at, kernels.cuh)
__device__ __forceinline__ int op_allele(const OpView& v, uint32_t off, uint32_t* q, int* ins) {
  *q = 0; *ins = 0;
  if (v.n == 0) return -1;
  uint32_t lo = 0, hi = v.n;
  while (lo < hi) { const uint32_t m = (lo + hi) >> 1; if (v.t[m] <= off) lo = m + 1; else hi = m; }
  const int k = (int)lo - 1;
  if (k < 0) return -1;
  int cnt = 0;
  for (int j = k; j >= 0 && v.t[j] == off; j--) cnt += ((v.w[j] & 3u) == HM_OP_INS);
  *ins = cnt;
  const uint32_t wd = v.w[k], kind = wd & 3u, val = wd >> 2, t0 = v.t[k];
  const uint32_t rl = (uint32_t)op_ref_len(wd);
  if (rl == 0 || off >= t0 + rl) return -1;
  if (kind == HM_OP_DEL) return 5;
  *q = v.q[k] + (kind == HM_OP_MATCH ? off - t0 : 0u);
  return kind == HM_OP_SUB ? (int)((val >> 3) & 7u) : 8;
}

// warp-cooperative: the chunk c with off[c] <= x < off[c + 1] (off: n + 1 ascending entries)
__device__ __forceinline__ uint32_t warp_find_chunk(const uint64_t* off, uint32_t n, uint64_t x, int lane) {
  uint32_t lo = 0, len = n + 1;
  while (len > 32) {
    const uint32_t step = (len + 32) / 33, end = lo + len;
    const uint32_t idx = lo + step * (uint32_t)(lane + 1) - 1;
    const bool below = idx < end && __ldg(off + idx) <= x;
    const uint32_t c = __popc(__ballot_sync(HM_FULL, below));
    lo += c * step;
    len = min(step, end - lo);
  }
  const bool below = (uint32_t)lane < len && __ldg(off + lo + lane) <= x;
  return lo + __popc(__ballot_sync(HM_FULL, below)) - 1;
}

// haplib.get_ccs_hap (haplib.py:61-83) for a warp over staged ops: lanes = hetSNPs
template <bool kSeq>
__device__ __forceinline__ int warp_read_hap_ops(const DevBatch& b, uint32_t r, int32_t ts, int32_t te, const OpView& v,
                                                 const DevPhase& ph, int set, int lane) {
  if (set < 0 || (uint32_t)set >= ph.n_sets) return 2;
  const uint64_t s0 = ph.set_off[set];
  const uint32_t n = (uint32_t)(ph.set_off[set + 1] - s0);
  const int32_t* hp = ph.hpos + s0;
  const uint32_t idx = upper_bound_dev(hp, n, ts);
  const uint32_t jdx = upper_bound_dev(hp, n, te);
  if (jdx - idx < 2) return 2;
  bool h0 = true, h1 = true;
  for (uint32_t k = idx + lane; k < jdx; k += 32) {
    uint32_t q; int ins;
    int a = op_allele(v, (uint32_t)(__ldg(hp + k) - 1 - ts), &q, &ins);
    const int hr = (int)ph.href[s0 + k];
    if (a == 8) a = kSeq ? (int)((b.seq[__ldg(b.seq_off + r) + (q >> 2)] >> (2 * (q & 3u))) & 3u) : href_match_base(hr);
    int bit = 2;
    if (a >= 0 && a < 4) {
      if (a == hr) bit = 0;
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

// ============================================================================ k_call_pairs
// One THREAD per (chunk, read) pair: a 15 kb CCS read is ~40 cs ops, a warp per pair leaves most lanes idle and the
// kernel is pure latency; with a thread per pair every pair of a 64 Mb contig is resident at once (one wave).
//
// pair_c[pr]: the pair's chunk, or 0xffffffff when the chunk does not fetch the read (k_call_scan starts from it).
// pair_hap (--phase only): 0 / 1 / 2 ("."), 3 = not fetched.
// num_ccs: a pair whose read passes the QV / MAPQ / identity / length gates and (--phase) has a haplotype marks the
//   read's query name; the first to mark a name counts it (m.num_ccs counts distinct names, caller.py:318-320).
// Candidates: the thread reserves one slot per substitution of its read in the chunk's segment (one atomic), fills
//   the slots of the substitutions that pass and marks the others as holes (HC_KEY_HOLE).
#define HC_KEY_HOLE 0xffffffffu

// haplib.get_ccs_hap for one thread over the read's ops (as thread_read_hap_walk, kernels.cuh), kSeq at compile time
template <bool kSeq>
__device__ __forceinline__ int thread_read_hap(const DevBatch& b, uint32_t r, int32_t ts, int32_t te, const uint32_t* ops, uint32_t nops,
                                               uint32_t qstart, const DevPhase& ph, int set) {
  if (set < 0 || (uint32_t)set >= ph.n_sets) return 2;
  const uint64_t s0 = ph.set_off[set];
  const uint32_t n = (uint32_t)(ph.set_off[set + 1] - s0);
  const int32_t* hp = ph.hpos + s0;
  const uint32_t idx = upper_bound_dev(hp, n, ts);
  const uint32_t jdx = upper_bound_dev(hp, n, te);
  if (jdx - idx < 2) return 2;
  uint32_t k = 0, t0 = 0, q0 = qstart;
  bool h0 = true, h1 = true;
  for (uint32_t i = idx; i < jdx; i++) {
    const uint32_t off = (uint32_t)(__ldg(hp + i) - 1 - ts);
    const int hr = (int)ph.href[s0 + i];
    int a = -1;
    while (k < nops) { // the op that holds reference offset `off`
      const uint32_t w = ops[k];
      const uint32_t rl = (uint32_t)op_ref_len(w);
      if (rl && off < t0 + rl) {
        const uint32_t kind = w & 3u, v = w >> 2;
        if (kind == HM_OP_DEL) a = 5;
        else if (kind == HM_OP_SUB) a = (int)((v >> 3) & 7u);
        else if (!kSeq) a = href_match_base(hr);
        else { const uint32_t q = q0 + (off - t0); a = (b.seq[__ldg(b.seq_off + r) + (q >> 2)] >> (2 * (q & 3u))) & 3; }
        break;
      }
      t0 += rl; q0 += (uint32_t)op_qry_len(w); k++;
    }
    int bit = 2;
    if (a >= 0 && a < 4) {
      if (a == hr) bit = 0;
      else if (a == (int)ph.halt[s0 + i]) bit = 1;
    }
    const int hb = ph.hbit[s0 + i];
    if (bit != hb) h0 = false;
    if (bit != 1 - hb) h1 = false;
  }
  return h0 ? 0 : (h1 ? 1 : 2);
}

#define HC_A_CAP 6144u // op words of a CTA's 128 reads staged in shared memory

// is op word w an entry of cs2subindel's mismatch list (cslib.py:47-64)?
__device__ __forceinline__ bool op_is_mismatch(uint32_t w) {
  const uint32_t kind = w & 3u;
  return kind == HM_OP_INS || kind == HM_OP_DEL || (kind == HM_OP_SUB && ((w >> 2) & 7u) != HM_BASE_N);
}

// largest c with off[c] <= x (off: n + 1 ascending entries, off[0] <= x < off[n]); 8-ary: three rounds of independent
// loads for a few hundred chunks instead of nine dependent ones
__device__ __forceinline__ uint32_t find_chunk_kary(const uint64_t* off, uint32_t n, uint64_t x) {
  uint32_t lo = 0, len = n + 1;
  while (len > 8) {
    const uint32_t step = (len + 7) >> 3, end = lo + len;
    uint32_t c = 0;
#pragma unroll
    for (uint32_t i = 1; i < 8; i++) {
      const uint32_t idx = lo + step * i - 1;
      if (idx < end) c += (__ldg(off + idx) <= x);
    }
    lo += c * step;
    len = min(step, end - lo);
  }
  uint32_t c = 0;
#pragma unroll
  for (uint32_t i = 0; i < 8; i++)
    if (i < len) c += (__ldg(off + lo + i) <= x);
  return lo + c - 1;
}

// the per-pair work of k_call_pairs once the read's ops are at hand; kShared: `ops` points into shared memory (the
// common case; a generic pointer would cost every load of the two walks an address-space check)
template <bool kSeq, bool kShared>
__device__ __forceinline__ void call_pair_body(const DevBatch& b, const DevParams& p, const DevPhase& ph, const uint32_t* ops_any,
                                               const hm_chunk& ch, uint32_t c, uint32_t r, uint64_t pr, uint32_t n, uint64_t o0,
                                               int32_t ts, int32_t te, int32_t qlen, uint32_t qstart, int mapq, uint8_t* pair_hap,
                                               uint32_t* qname_seen32, unsigned long long* num_ccs, const uint64_t* seg_off, uint32_t* seg_cnt,
                                               uint32_t* seg_keys, uint32_t* seg_read) {
  struct Ops { // address-space-specific loads; the shared window address is taken once
    const uint32_t* p;
    uint32_t sbase;
    __device__ __forceinline__ uint32_t operator[](uint32_t k) const {
      if (kShared) { uint32_t v; asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(sbase + 4u * k)); return v; }
      return __ldg(p + k);
    }
  };
  const Ops ops = {ops_any, kShared ? (uint32_t)__cvta_generic_to_shared(ops_any) : 0u};

  // walk 1, branch-free per op: identity tallies (bamlib.get_blast_sequence_identity), substitutions inside the chunk;
  // op prefixes to HBM for the op lists k_call_scan does not stage itself
  uint32_t t = 0;
  int nm = 0, ns = 0, il = 0, dl = 0, n_sub_in = 0;
  const bool long_ops = n > HC_MAX_OPS;
  uint32_t qq = qstart;
  const int32_t lo_t = ch.start - ts - 1, hi_t = ch.end - ts - 1; // candidate <=> lo_t <= t <= hi_t (tpos = ts + t + 1)
  for (uint32_t k0 = 0; k0 < n; k0 += 4) { // four ops per round: their loads go out together (a zero word is an empty match run)
    uint32_t w4[4];
#pragma unroll
    for (uint32_t u = 0; u < 4; u++) w4[u] = k0 + u < n ? ops[k0 + u] : 0u;
#pragma unroll
    for (uint32_t u = 0; u < 4; u++) {
      const uint32_t w = w4[u];
      const uint32_t kind = w & 3u, v = w >> 2;
      if (long_ops && k0 + u < n) { b.op_t[o0 + k0 + u] = t; b.op_q[o0 + k0 + u] = qq; qq += (uint32_t)op_qry_len(w); }
      const bool is_m = kind == HM_OP_MATCH, is_s = kind == HM_OP_SUB, is_i = kind == HM_OP_INS, is_d = kind == HM_OP_DEL;
      nm += is_m ? (int)v : 0; ns += is_s; il += is_i ? (int)v : 0; dl += is_d ? (int)v : 0;
      n_sub_in += (is_s && (v & 7u) != HM_BASE_N && (int32_t)t >= lo_t && (int32_t)t <= hi_t);
      t += (is_m || is_d) ? v : (uint32_t)is_s;
    }
  }

  // read gates of caller.py:310-317, same order of evaluation; the QV gate is bamlib.get_qv (np.mean of the read's
  // qualities: the resident integer sum divided once)
  bool pre_ok = true;
  if (__ddiv_rn((double)__ldg(b.bq_total + r), (double)qlen) < (double)p.min_qv) pre_ok = false;
  if (mapq < p.min_mapq) pre_ok = false;
  const double ident = __ddiv_rn((double)nm, (double)(nm + ns + il + dl));
  if (ident < p.min_sequence_identity) pre_ok = false;
  if (!(p.qlen_lower_limit < qlen && qlen < p.qlen_upper_limit)) pre_ok = false;
  if (p.phase) {
    const int hap = thread_read_hap<kSeq>(b, r, ts, te, ops_any, n, qstart, ph, ch.phase_set);
    pair_hap[pr] = (uint8_t)hap;
    if (hap > 1) return;
  }
  if (!pre_ok) return;
  { // one byte per query name, set through 32-bit atomics
    const uint32_t qn = __ldg(b.qname_id + r);
    const uint32_t bit = 1u << (8u * (qn & 3u));
    if (!(atomicOr(qname_seen32 + (qn >> 2), bit) & bit)) atomicAdd(num_ccs + (r & 7u), 1ull);
  }
  if (n_sub_in == 0) return;

  // walk 2: bamlib.get_tsbs_candidates (bamlib.py:69-86) for every substitution of the read that lies in the chunk.
  // A lane first runs ahead to its next such substitution (a short loop), then the lanes of the warp test theirs
  // together.  The mismatch-window count (bamlib.py:266-282: entries of the sorted mismatch list inside
  // [tpos - u, tpos + d], minus the substitution itself) is taken from the neighbouring ops directly — every non-match
  // op is one entry of that list (cs2subindel), at the reference position the walk has reached — and stops as soon
  // as it exceeds max_mismatch_count.
  const uint64_t slot0 = __ldg(seg_off + c) + atomicAdd(seg_cnt + c, (uint32_t)n_sub_in);
  const double trim_s = floor(__dmul_rn(p.min_trim, (double)qlen));
  const double trim_e = ceil(__dmul_rn(__dsub_rn(1.0, p.min_trim), (double)qlen));
  const int wsz = p.mismatch_window, max_mm = p.max_mismatch_count;
  uint32_t q = qstart, k = 0;
  t = 0;
  for (int used = 0; used < n_sub_in; used++) {
    uint32_t w = 0;
    for (; k < n; k++) { // to the next substitution inside the chunk
      w = ops[k];
      const uint32_t kind = w & 3u, v = w >> 2;
      if (kind == HM_OP_SUB && (v & 7u) != HM_BASE_N && (int32_t)t >= lo_t && (int32_t)t <= hi_t) break;
      t += (kind == HM_OP_MATCH || kind == HM_OP_DEL) ? v : (uint32_t)(kind == HM_OP_SUB);
      q += (kind == HM_OP_MATCH || kind == HM_OP_INS) ? v : (uint32_t)(kind == HM_OP_SUB);
    }
    if (k >= n) break; // cannot happen: walk 1 counted n_sub_in of them
    const uint32_t v = w >> 2;
    const int32_t tpos = ts + (int32_t)t + 1;
    const int32_t qpos = (int32_t)q;
    uint32_t key = HC_KEY_HOLE;
    if (!((double)qpos < trim_s) && !((double)qpos > trim_e)) {
      const int qs = qpos - wsz, qe = qpos + wsz; // bamlib.get_mismatch_range
      int u, d;
      if (qs < 0) { u = wsz + qs; d = wsz + (-qs); }
      else if (qe > qlen) { u = wsz + (qe - qlen); d = qlen - qpos; }
      else { u = wsz; d = wsz; }
      int cnt = 0;
      uint32_t tj = t + 1; // reference offset at the start of op k + 1
      for (uint32_t j = k + 1; j < n && cnt <= max_mm; j++) { // later entries of the list, ascending positions
        const uint32_t wj = ops[j];
        if (ts + (int32_t)tj + 1 > tpos + d) break; // nothing from here on can be inside the window
        cnt += op_is_mismatch(wj);
        tj += (uint32_t)op_ref_len(wj);
      }
      tj = t; // reference offset at the start of op k
      for (uint32_t j = k; j-- > 0 && cnt <= max_mm;) { // earlier entries, descending positions
        const uint32_t wj = ops[j];
        tj -= (uint32_t)op_ref_len(wj); // offset at the start of op j
        if (op_is_mismatch(wj)) {
          if (ts + (int32_t)tj + 1 < tpos - u) break;
          cnt++;
        } else if (ts + (int32_t)tj + 1 < tpos - u) break; // a match run that starts before the window: nothing earlier counts
      }
      if (!(cnt > max_mm)) key = ((uint32_t)(tpos - ch.start) << 4) | ((v & 3u) << 2) | ((v >> 3) & 3u);
    }
    seg_keys[slot0 + used] = key;
    seg_read[slot0 + used] = r;
    t += 1; q += 1; k++;
  }
}

template <bool kSeq>
__global__ void __launch_bounds__(128) k_call_pairs(DevBatch b, DevParams p, DevPhase ph, const hm_chunk* chunks, uint32_t n_chunks,
                                                    const uint64_t* pair_off, uint64_t n_pairs, uint32_t* pair_c, uint8_t* pair_hap,
                                                    uint32_t* qname_seen32, unsigned long long* num_ccs, const uint64_t* seg_off,
                                                    uint32_t* seg_cnt, uint32_t* seg_keys, uint32_t* seg_read) {
  extern __shared__ uint32_t s_ops[]; // HC_A_CAP
  __shared__ unsigned long long s_span[2];
  if (threadIdx.x == 0) { s_span[0] = ~0ull; s_span[1] = 0ull; }
  __syncthreads();
  const uint64_t pr = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool active = pr < n_pairs;
  uint32_t c = 0, r = 0, n = 0, qstart = 0;
  hm_chunk ch = {0, 0, 0, 0, 0, 0};
  int32_t ts = 0, te = 0, qlen = 0;
  uint64_t o0 = 0;
  int mapq = 0;
  if (active) {
    c = find_chunk_kary(pair_off, n_chunks, pr);
    ch = chunks[c];
    r = ch.read_lo + (uint32_t)(pr - __ldg(pair_off + c));
    // everything the pair needs from the read, loaded together
    const uint32_t flags = __ldg(b.flags + r);
    ts = __ldg(b.tstart + r); te = __ldg(b.tend + r);
    n = __ldg(b.n_ops + r);
    o0 = __ldg(b.op_off + r);
    qlen = __ldg(b.qlen + r);
    qstart = (uint32_t)__ldg(b.qstart + r);
    mapq = (int)__ldg(b.mapq + r);
    if ((flags & HM_READ_SECONDARY) || !(ts < ch.end && te > ch.start)) {
      pair_c[pr] = 0xffffffffu;
      if (p.phase) pair_hap[pr] = 3;
      active = false;
    } else {
      pair_c[pr] = c;
    }
  }
  { // the run of the op stream this CTA's reads span: warp reduction, one shared atomic per warp
    unsigned long long lo = (active && n) ? (unsigned long long)o0 : ~0ull, hi = (active && n) ? (unsigned long long)(o0 + n) : 0ull;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      const unsigned long long a = __shfl_xor_sync(HM_FULL, lo, d), e = __shfl_xor_sync(HM_FULL, hi, d);
      lo = min(lo, a); hi = max(hi, e);
    }
    if ((threadIdx.x & 31) == 0) { atomicMin(&s_span[0], lo); atomicMax(&s_span[1], hi); }
  }
  __syncthreads();
  // the CTA's reads are neighbours in the file, so their ops are one short run of the op stream: staged with
  // coalesced loads (a thread walking its own ops in global memory costs one L1 wavefront per lane and load)
  const unsigned long long sp_lo = s_span[0], sp_hi = s_span[1];
  const bool staged = sp_hi > sp_lo && sp_hi - sp_lo <= HC_A_CAP;
  if (staged) { // eight independent loads per thread and round: the run is ~40 words per thread, one round trip each otherwise
    const uint32_t nw = (uint32_t)(sp_hi - sp_lo);
    const uint32_t* src = b.ops + sp_lo;
    for (uint32_t i0 = threadIdx.x; i0 < nw; i0 += 8 * blockDim.x) {
      uint32_t v[8];
#pragma unroll
      for (int u = 0; u < 8; u++) { const uint32_t i = i0 + u * blockDim.x; v[u] = i < nw ? __ldg(src + i) : 0u; }
#pragma unroll
      for (int u = 0; u < 8; u++) { const uint32_t i = i0 + u * blockDim.x; if (i < nw) s_ops[i] = v[u]; }
    }
  }
  __syncthreads();
  if (!active) return;
  if (staged)
    call_pair_body<kSeq, true>(b, p, ph, s_ops + (o0 - sp_lo), ch, c, r, pr, n, o0, ts, te, qlen, qstart, mapq, pair_hap, qname_seen32, num_ccs,
                               seg_off, seg_cnt, seg_keys, seg_read);
  else
    call_pair_body<kSeq, false>(b, p, ph, b.ops + o0, ch, c, r, pr, n, o0, ts, te, qlen, qstart, mapq, pair_hap, qname_seen32, num_ccs,
                                seg_off, seg_cnt, seg_keys, seg_read);
}

// ============================================================================ k_site_sort
// block-wide exclusive scan of one value per thread (HC_SORT_THREADS threads); returns the exclusive prefix, *total
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t* s_warp, uint32_t* total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(HM_FULL, incl, d); if (lane >= d) incl += t; }
  __syncthreads(); // s_warp may still be read from a previous scan
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    uint32_t w = lane < (int)(blockDim.x >> 5) ? s_warp[lane] : 0u, wi = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(HM_FULL, wi, d); if (lane >= d) wi += t; }
    s_warp[lane] = wi - w;        // exclusive prefix of the warp totals
    if (lane == 31) s_warp[32] = wi; // grand total
  }
  __syncthreads();
  *total = s_warp[32];
  return s_warp[wid] + incl - v;
}

// One CTA per tile.  tile_chunk[t] = chunk of tile t, tile_off[c] = first tile of chunk c (host).  Outputs: the
// tile's sorted distinct keys (chunk-relative: rel << 4 | ref << 2 | alt) at keys_tmp[tile_src[t] ...) and tile_cnt[t].
// The tile's own keys are staged in shared memory once (the chunk's segment is read a single time, coalesced); a tile
// with more keys than the stage holds walks the segment in global memory instead.
#define HC_STAGE 8192u
__global__ void __launch_bounds__(HC_SORT_THREADS) k_site_sort(const uint32_t* tile_chunk, const uint32_t* tile_off, const uint64_t* seg_off,
                                                               const uint32_t* seg_cnt, const uint32_t* seg_keys, uint32_t* chunk_cursor,
                                                               uint32_t* chunk_cursor2, uint32_t* gscratch, uint32_t* keys_tmp,
                                                               uint32_t* tile_src, uint32_t* tile_cnt) {
  extern __shared__ uint32_t sm[];
  uint32_t* s_bits = sm;                          // HC_TILE_WORDS
  uint32_t* s_wpre = s_bits + HC_TILE_WORDS;      // HC_TILE_WORDS: distinct positions before each word
  uint32_t* s_mask = s_wpre + HC_TILE_WORDS;      // HC_CAPD: (ref, alt) combinations seen at the rank-th distinct position
  uint32_t* s_off = s_mask + HC_CAPD;             // HC_CAPD: distinct keys before the rank-th distinct position
  uint32_t* s_keys = s_off + HC_CAPD;             // HC_STAGE: the tile's keys
  __shared__ uint32_t s_warp[33];
  __shared__ uint32_t s_base[2];
  __shared__ uint32_t s_nstaged;
  const uint32_t t = blockIdx.x, tid = threadIdx.x;
  const uint32_t c = tile_chunk[t];
  const uint32_t tile_in_chunk = t - tile_off[c];
  const uint64_t seg0 = seg_off[c];
  const uint32_t nk = seg_cnt[c];
  const uint32_t* keys = seg_keys + seg0;

  for (uint32_t i = tid; i < HC_TILE_WORDS; i += blockDim.x) s_bits[i] = 0u;
  if (tid == 0) s_nstaged = 0;
  __syncthreads();
  // position bitmap; the tile's keys go to the stage as long as they fit (holes: slots of substitutions that failed)
  for (uint32_t j0 = 0; j0 < nk; j0 += 4 * blockDim.x) {
    uint32_t kv[4];
#pragma unroll
    for (int u = 0; u < 4; u++) { const uint32_t j = j0 + u * blockDim.x + tid; kv[u] = j < nk ? __ldg(keys + j) : HC_KEY_HOLE; }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const uint32_t rel = kv[u] >> 4;
      if (kv[u] == HC_KEY_HOLE || (rel >> HC_TILE_BITS) != tile_in_chunk) continue;
      atomicOr(&s_bits[(rel & (HC_TILE - 1u)) >> 5], 1u << (rel & 31u));
      const uint32_t at = atomicAdd(&s_nstaged, 1u);
      if (at < HC_STAGE) s_keys[at] = kv[u];
    }
  }
  __syncthreads();
  const uint32_t n_own = s_nstaged;
  const bool staged = n_own <= HC_STAGE;
  // distinct positions before each bitmap word: each thread owns HC_TILE_WORDS / blockDim.x consecutive words
  constexpr uint32_t WPT = HC_TILE_WORDS / HC_SORT_THREADS;
  uint32_t local = 0;
#pragma unroll
  for (uint32_t i = 0; i < WPT; i++) local += __popc(s_bits[tid * WPT + i]);
  uint32_t n_dist;
  uint32_t run = block_excl_scan(local, s_warp, &n_dist);
#pragma unroll
  for (uint32_t i = 0; i < WPT; i++) { s_wpre[tid * WPT + i] = run; run += __popc(s_bits[tid * WPT + i]); }
  // (ref, alt) masks and offsets per distinct position: shared memory, or this tile's own piece of the global scratch
  const bool in_smem = n_dist <= HC_CAPD;
  if (!in_smem && tid == 0) s_base[0] = atomicAdd(chunk_cursor2 + c, 2u * n_dist); // n_dist <= keys of the tile
  __syncthreads();
  uint32_t* mask = in_smem ? s_mask : gscratch + 2 * seg0 + s_base[0];
  uint32_t* off = in_smem ? s_off : mask + n_dist;
  for (uint32_t i = tid; i < n_dist; i += blockDim.x) mask[i] = 0u;
  __syncthreads();
  const uint32_t n_walk = staged ? n_own : nk;
  const uint32_t* walk = staged ? s_keys : keys;
  for (uint32_t j = tid; j < n_walk; j += blockDim.x) {
    const uint32_t key = walk[j], rel = key >> 4;
    if (key == HC_KEY_HOLE || (rel >> HC_TILE_BITS) != tile_in_chunk) continue;
    const uint32_t p = rel & (HC_TILE - 1u);
    const uint32_t rank = s_wpre[p >> 5] + __popc(s_bits[p >> 5] & ((1u << (p & 31u)) - 1u));
    atomicOr(&mask[rank], 1u << (key & 15u));
  }
  __syncthreads();
  // distinct keys before each distinct position: each thread owns a consecutive run of ranks
  const uint32_t per = (n_dist + blockDim.x - 1) / blockDim.x;
  const uint32_t r0 = min(tid * per, n_dist), r1 = min(r0 + per, n_dist);
  local = 0;
  for (uint32_t i = r0; i < r1; i++) local += __popc(mask[i]);
  uint32_t n_uniq;
  run = block_excl_scan(local, s_warp, &n_uniq);
  for (uint32_t i = r0; i < r1; i++) { off[i] = run; run += __popc(mask[i]); }
  if (tid == 0) {
    const uint32_t at = atomicAdd(chunk_cursor + c, n_uniq); // tiles of a chunk share its segment of keys_tmp
    s_base[1] = at;
    tile_src[t] = (uint32_t)seg0 + at;
    tile_cnt[t] = n_uniq;
  }
  __syncthreads();
  uint32_t* dst = keys_tmp + seg0 + s_base[1];
  // sorted distinct keys: positions ascending (bitmap order), then (ref, alt) ascending (mask bit order)
#pragma unroll 1
  for (uint32_t i = 0; i < WPT; i++) {
    const uint32_t wi = tid * WPT + i;
    uint32_t bits = s_bits[wi];
    uint32_t rank = s_wpre[wi];
    while (bits) {
      const uint32_t bit = __ffs(bits) - 1;
      bits &= bits - 1;
      uint32_t m = mask[rank], o = off[rank];
      const uint32_t rel = (tile_in_chunk << HC_TILE_BITS) | (wi << 5) | bit;
      while (m) { const uint32_t cb = __ffs(m) - 1; m &= m - 1; dst[o++] = (rel << 4) | cb; }
      rank++;
    }
  }
}

// exclusive scan of tile_cnt -> tile_dst[0 .. n_tiles]; cnt[1] = number of distinct sites, or 0 with cnt[5] = the
// number needed when it exceeds site_cap (the host grows its buffers and runs the call again)
__global__ void __launch_bounds__(1024) k_tile_scan(const uint32_t* tile_cnt, uint32_t n_tiles, uint32_t* tile_dst, unsigned long long site_cap,
                                                    unsigned long long* cnt) {
  __shared__ uint32_t s_warp[33];
  uint32_t carry = 0;
  for (uint32_t base = 0; base < n_tiles; base += blockDim.x) {
    const uint32_t i = base + threadIdx.x;
    const uint32_t v = i < n_tiles ? tile_cnt[i] : 0u;
    uint32_t total;
    const uint32_t ex = block_excl_scan(v, s_warp, &total);
    if (i < n_tiles) tile_dst[i] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0) {
    const bool over = (unsigned long long)carry > site_cap;
    tile_dst[n_tiles] = over ? 0u : carry;
    cnt[1] = over ? 0ull : (unsigned long long)carry;
    cnt[5] = over ? (unsigned long long)carry : 0ull;
  }
  if (n_tiles == 0 && threadIdx.x == 0) tile_dst[0] = 0u;
}

// final key array (chunk << 36 | tpos << 4 | ref << 2 | alt, sorted), the file-order read range of every site
// (as k_site_range), its entry slots set to "unwritten"
__global__ void __launch_bounds__(256) k_site_range2(DevBatch b, const hm_chunk* chunks, const uint32_t* tile_chunk, const uint32_t* tile_src,
                                                     const uint32_t* tile_dst, uint32_t n_tiles, const uint32_t* keys_tmp,
                                                     const unsigned long long* n_keys_dev, unsigned long long* keys, uint32_t* site_lo,
                                                     uint32_t* site_n, uint32_t* entries, uint64_t stride, uint32_t n_slots) {
  const uint64_t ki = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (ki >= *n_keys_dev) return;
  const uint32_t t = upper_bound_dev(tile_dst, n_tiles + 1, (uint32_t)ki) - 1; // last tile with tile_dst <= ki (empty tiles repeat a value)
  const uint32_t c = __ldg(tile_chunk + t);
  const hm_chunk ch = chunks[c];
  const uint32_t k32 = __ldg(keys_tmp + __ldg(tile_src + t) + ((uint32_t)ki - __ldg(tile_dst + t)));
  const int32_t tpos = ch.start + (int32_t)(k32 >> 4);
  keys[ki] = ((unsigned long long)c << 36) | ((unsigned long long)(uint32_t)tpos << 4) | (unsigned long long)(k32 & 15u);
  const int32_t rpos = tpos - 1;
  const uint32_t n_in = ch.read_hi - ch.read_lo;
  const uint32_t lo = count_le_kary_i32(b.pmax_tend + ch.read_lo, n_in, rpos - 1);
  const uint32_t hi = count_le_kary_i32(b.tstart + ch.read_lo, n_in, rpos);
  const uint32_t n = hi > lo ? hi - lo : 0u;
  site_lo[ki] = ch.read_lo + lo;
  site_n[ki] = n;
  const uint32_t ns = min(n, n_slots);
  for (uint32_t s = 0; s < ns; s++) entries[(uint64_t)s * stride + ki] = HM_ENT_UNWRITTEN;
}

// ============================================================================ k_call_scan
// One warp per (chunk, read) pair, HC_SCAN_WARPS warps per CTA.  The warp finds the chunk's sites the read can touch,
// stages the read's ops with their prefixes in shared memory, lists the first HC_SITES sites in registers (entry
// without its quality, query position of the base, entry address) and then fetches their quality bytes, every load
// of the list issued before any of its entries is written.  The QV gate is k_call_pairs' (the resident quality sum):
// nothing here streams the qualities, a lookup costs one sector of the stream.
#ifndef HC_SCAN_WARPS
#define HC_SCAN_WARPS 4
#endif
#ifndef HC_SITES
#define HC_SITES 64 // sites of a pair kept in the list (registers); the rest go the direct way
#endif
#ifndef HC_SCAN_MINB
#define HC_SCAN_MINB 10 // resident CTAs per SM asked of the compiler (register budget)
#endif

struct __align__(16) ScanWarp {
  uint32_t w[HC_MAX_OPS], t[HC_MAX_OPS], q[HC_MAX_OPS];
};

template <bool kSeq>
__global__ void __launch_bounds__(32 * HC_SCAN_WARPS, HC_SCAN_MINB) k_call_scan(DevBatch b, DevParams p, const hm_chunk* chunks, const uint64_t* pair_off,
                                                                  uint64_t n_pairs, const uint32_t* pair_c, const uint8_t* pair_hap,
                                                                  const uint32_t* tile_off, const uint32_t* tile_dst,
                                                                  const unsigned long long* keys, const uint32_t* site_lo,
                                                                  const uint32_t* site_n, uint32_t* entries, uint32_t stride,
                                                                  const unsigned long long* n_keys_dev, uint32_t n_slots) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  const uint64_t pr = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (pr >= n_pairs) return;
  const uint32_t c = __ldg(pair_c + pr);
  if (c == 0xffffffffu) return; // the chunk does not fetch the read
  if (*n_keys_dev == 0) return; // no sites (also when the site list overflowed its buffers: the host runs the call again)
  ScanWarp* S = reinterpret_cast<ScanWarp*>(smem_raw) + wid;
  const uint32_t to0 = __ldg(tile_off + c), to1 = __ldg(tile_off + c + 1);
  const uint32_t r = __ldg(&chunks[c].read_lo) + (uint32_t)(pr - __ldg(pair_off + c));
  const int32_t ts = __ldg(b.tstart + r), te = __ldg(b.tend + r);
  const uint32_t n = __ldg(b.n_ops + r);
  const uint32_t k_lo = __ldg(tile_dst + to0), k_hi = __ldg(tile_dst + to1);
  if (n == 0 || k_lo >= k_hi) return;

  // the chunk's sites the read can touch: rpos in [ts, te], i.e. tpos in [ts + 1, te + 1]
  const unsigned long long kb = (unsigned long long)c << 36;
  const uint32_t s_lo = warp_lower_bound_u64(keys, k_lo, k_hi, kb | ((unsigned long long)(uint32_t)(ts + 1) << 4), lane);
  const uint32_t s_hi = warp_lower_bound_u64(keys, s_lo, k_hi, kb | ((unsigned long long)(uint32_t)(te + 2) << 4), lane);
  if (s_lo >= s_hi) return;
  const uint64_t o0 = __ldg(b.op_off + r);
  const uint8_t* bqg = b.bq + __ldg(b.bq_off + r);
  const uint32_t qlen = (uint32_t)__ldg(b.qlen + r);
  const uint32_t hap = p.phase ? (uint32_t)__ldg(pair_hap + pr) : 2u;
  const bool staged = n <= HC_MAX_OPS;
  if (staged) { // the prefix scan again (registers only): cheaper than keeping 8 B per op in HBM
    uint32_t t_carry = 0, q_carry = (uint32_t)__ldg(b.qstart + r);
    for (uint32_t base = 0; base < n; base += 32) {
      const uint32_t k = base + lane;
      const uint32_t w = k < n ? __ldg(b.ops + o0 + k) : 0u;
      const uint32_t rl = (uint32_t)op_ref_len(w), al = (uint32_t)op_qry_len(w);
      uint32_t rs = rl, qs = al;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t a = __shfl_up_sync(HM_FULL, rs, d), e = __shfl_up_sync(HM_FULL, qs, d);
        if (lane >= d) { rs += a; qs += e; }
      }
      if (k < n) { S->w[k] = w; S->t[k] = t_carry + rs - rl; S->q[k] = q_carry + qs - al; }
      t_carry += __shfl_sync(HM_FULL, rs, 31);
      q_carry += __shfl_sync(HM_FULL, qs, 31);
    }
    __syncwarp();
  }
  const OpView view = {staged ? S->w : b.ops + o0, staged ? S->t : b.op_t + o0, staged ? S->q : b.op_q + o0, n};
  const uint64_t sq0 = kSeq ? __ldg(b.seq_off + r) : 0;

  // one site: entry without its quality, the query position of the base (0xffffffff: the site needs no quality byte
  // of this read, its entry is written at once), the entry's address
  auto site = [&](uint32_t ki, uint32_t* q_out, uint32_t* e_out, uint32_t* at_out) {
    *q_out = 0xffffffffu; *e_out = 0; *at_out = 0;
    const uint32_t slot = r - __ldg(site_lo + ki);
    if (slot >= n_slots || slot >= __ldg(site_n + ki)) return; // pileups deeper than the slots: k_site_reduce computes these itself
    const unsigned long long key = __ldg(keys + ki);
    const int32_t rpos = (int32_t)((key >> 4) & 0xffffffffull) - 1;
    uint32_t q; int ins;
    int a = op_allele(view, (uint32_t)(rpos - ts), &q, &ins);
    const bool has_base = a >= 0 && a != 5;
    if (a == 8) a = kSeq ? (int)((b.seq[sq0 + (q >> 2)] >> (2 * (q & 3u))) & 3u) : (int)((key >> 2) & 3);
    const uint32_t e = (a < 0 ? HM_ENT_NONE : (uint32_t)a) | ((uint32_t)min(ins, 255) << 11) | ((hap & 3u) << 19) |
                       ((te > rpos + 1) ? (1u << 21) : 0u);
    const uint32_t at = slot * stride + ki;
    if (has_base) { *q_out = q; *e_out = e; *at_out = at; }
    else entries[at] = e;
  };
  // the quality byte of query position q (0 past the read's end: malformed ops)
  auto qual = [&](uint32_t q) { return q < qlen ? (uint32_t)__ldg(bqg + q) : 0u; };

  // the pair's site list (the first HC_SITES sites), HC_SITES / 32 per lane, in registers
  const uint32_t n_list = min(s_hi - s_lo, (uint32_t)HC_SITES);
  uint32_t lq[HC_SITES / 32], le[HC_SITES / 32], la[HC_SITES / 32];
#pragma unroll
  for (uint32_t g = 0; g < HC_SITES / 32; g++) {
    const uint32_t i = g * 32 + (uint32_t)lane;
    lq[g] = 0xffffffffu; le[g] = 0; la[g] = 0;
    if (i < n_list) site(s_lo + i, &lq[g], &le[g], &la[g]);
  }
  uint32_t lb[HC_SITES / 32];
#pragma unroll
  for (uint32_t g = 0; g < HC_SITES / 32; g++) lb[g] = lq[g] != 0xffffffffu ? qual(lq[g]) : 0u;
#pragma unroll
  for (uint32_t g = 0; g < HC_SITES / 32; g++)
    if (lq[g] != 0xffffffffu) entries[la[g]] = le[g] | (lb[g] << 3);
  // sites past the list: the direct way
  for (uint32_t k0 = s_lo + HC_SITES; k0 < s_hi; k0 += 32) {
    const uint32_t ki = k0 + (uint32_t)lane;
    if (ki >= s_hi) continue;
    uint32_t q, e, at;
    site(ki, &q, &e, &at);
    if (q != 0xffffffffu) entries[at] = e | (qual(q) << 3);
  }
}

// ============================================================================ k_publish_call
// Everything the host reads at the one synchronisation of a call, in one launch, into mapped pinned memory:
// the counters and the first boundary records (index in key order, position among the kept records, the record).
__global__ void __launch_bounds__(256) k_publish_call(const uint32_t* cnt, uint32_t cnt_words, const uint32_t* bidx, const uint32_t* bpos,
                                                      const uint32_t* brecs, uint32_t max_items, const unsigned long long* n_items_dev,
                                                      uint32_t* m_cnt, uint32_t* m_bidx, uint32_t* m_bpos, uint32_t* m_brecs) {
  const uint32_t n = (uint32_t)min((unsigned long long)max_items, *n_items_dev);
  const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
  for (uint32_t i = tid; i < cnt_words; i += nth) m_cnt[i] = cnt[i];
  for (uint32_t i = tid; i < n; i += nth) { m_bidx[i] = bidx[i]; m_bpos[i] = bpos[i]; }
  const uint32_t rw = (uint32_t)(sizeof(hm_site_record) / 4);
  for (uint32_t i = tid; i < n * rw; i += nth) m_brecs[i] = brecs[i];
  __threadfence_system();
}
