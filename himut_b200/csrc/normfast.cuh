// normfast.cuh — exact pass of the callable-base half of `himut normcounts` on sm_100a
// (normcounts.get_callable_tricounts, src/himut/normcounts.py:240-419), and `himut phase` edge counting.
//
// The integer pass in front of it (k_norm_bits, normbits.cuh) settles every pure position whose verdict is certified
// and lists the others (about 1-2 % of the positions) as sites:
//
//   k_norm_site_range   per site: the file-order range of the chunk's reads that can touch it;
//   k_norm_entries_bits (normbits.cuh) gathers the pileup column, one warp per (chunk, read); a read it cannot
//                       stage is answered by norm_entry;
//   k_norm_reduce       per site in file order: the ordered fp64 sums, ten PL, argmin, GQ and the cascade exactly as
//                       k_norm_tiles_tma does it.
//
// Both passes add into the same NormOut tallies, so the result is bit-identical to evaluating every position exactly
// (k_norm_tiles_tma, normcounts.cuh, which runs instead where the bit vectors do not apply: parameters outside the
// certified domain, a chunk that starts below position 0, 2^32 or more cal words in one batch).
#pragma once
#include "normcounts.cuh"

// ============================================================================ exact pass
// entry: bits 0-2 allele (0-3 base, 5 deleted, 7 none), 3-10 BQ, 11-18 insertions at the site,
//        19-20 haplotype (0, 1, 2 "."), 21 counted by update_tri2count (read passes its gates too)
__device__ __forceinline__ uint32_t norm_entry(const DevBatch& b, const DevParams& p, const hm_chunk& ch, uint32_t pf, uint32_t r,
                                               int32_t pos) {
  if (!(pf & HM_PF_FETCHED)) return HM_ENT_NONE;
  const int32_t ts = __ldg(b.tstart + r), te = __ldg(b.tend + r);
  if (!(ts < ch.end && te > ch.start && ts <= pos && pos <= te)) return HM_ENT_NONE;
  const uint32_t n = __ldg(b.n_ops + r);
  if (n == 0) return HM_ENT_NONE;
  const uint64_t o0 = __ldg(b.op_off + r);
  const uint32_t off = (uint32_t)(pos - ts);
  const int k = (int)count_le_kary(b.op_t + o0, n, off) - 1;
  int ins = 0;
  for (int j = k; j >= 0 && __ldg(b.op_t + o0 + j) == off; j--)
    if ((__ldg(b.ops + o0 + j) & 3u) == HM_OP_INS) ins++;
  const uint32_t wd = __ldg(b.ops + o0 + k);
  const uint32_t kind = wd & 3u, t_op = __ldg(b.op_t + o0 + k), q0 = __ldg(b.op_q + o0 + k);
  const uint32_t rl = (uint32_t)op_ref_len(wd);
  uint32_t a = HM_ENT_NONE, bq = 0, cnt = 0;
  if (rl != 0 && off < t_op + rl) {
    if (kind == HM_OP_DEL) a = 5u;
    else {
      const uint32_t q = q0 + (kind == HM_OP_MATCH ? off - t_op : 0u);
      bq = b.bq[__ldg(b.bq_off + r) + q];
      a = kind == HM_OP_SUB ? ((wd >> 5) & 3u) : (uint32_t)((b.seq[__ldg(b.seq_off + r) + (q >> 2)] >> (2 * (q & 3u))) & 3u);
      if (pf & HM_PF_PASS) {
        if (kind == HM_OP_SUB) cnt = 1;                       // normcounts.py:95-108: always counted
        else if ((int)bq >= p.min_bq) {
          const int32_t qlen = __ldg(b.qlen + r);
          const int32_t trim_s = (int32_t)floor(__dmul_rn(p.min_trim, (double)qlen));
          const int32_t trim_e = (int32_t)ceil(__dmul_rn(__dsub_rn(1.0, p.min_trim), (double)qlen));
          if (!((int32_t)q < trim_s || (int32_t)q > trim_e)) {
            const int w = p.mismatch_window;
            const int32_t qpos0 = (int32_t)q0;
            const int qs = qpos0 - w, qe = qpos0 + w;
            int u, d;
            if (qs < 0) { u = w + qs; d = w + (-qs); }
            else if (qe > qlen) { u = w + (qe - qlen); d = qlen - qpos0; }
            else { u = w; d = w; }
            const int32_t* mm = b.mm_pos + o0;
            const uint32_t nmm = (uint32_t)__ldg(b.n_mm + r);
            const int mc = (int)count_le_kary_i32(mm, nmm, pos + d) - (int)count_le_kary_i32(mm, nmm, pos - u - 1);
            cnt = !(mc > p.max_mismatch_count);
          }
        }
      }
    }
  }
  return a | (bq << 3) | ((uint32_t)min(ins, 255) << 11) | (((pf >> HM_PF_HAP_SHIFT) & 3u) << 19) | (cnt << 21);
}

// kTrack: a counted site also stores its callable count into the track (track_at, normcounts.cuh)
template <bool kTrack>
__global__ void __launch_bounds__(128) k_norm_reduce(DevBatch b, DevParams p, DevSets sets, DevLut lut, const hm_chunk* chunks,
                                                     const uint64_t* pair_off, const uint8_t* pair_flag,
                                                     const unsigned long long* keys, uint64_t n_keys, const uint32_t* site_lo,
                                                     const uint32_t* site_n, const uint32_t* entries, uint64_t stride,
                                                     const uint8_t* refseq, uint64_t ref_len, NormOut* out, uint32_t n_slots,
                                                     uint32_t* track, const uint64_t* track_off) {
  __shared__ double s_lut[3][256];
  __shared__ unsigned long long s_ccs[HM_TRI_BINS], s_ref[HM_TRI_BINS], s_log[HM_NORM_LOG_LEN], s_tie;
  __shared__ int s_err;
  for (int i = threadIdx.x; i < 768; i += blockDim.x) s_lut[i >> 8][i & 255] = __ldg(lut.lut + i);
  if (threadIdx.x < HM_TRI_BINS) { s_ccs[threadIdx.x] = 0; s_ref[threadIdx.x] = 0; }
  if (threadIdx.x < HM_NORM_LOG_LEN) s_log[threadIdx.x] = 0;
  if (threadIdx.x == 0) { s_tie = 0; s_err = 0; }
  __syncthreads();
  const uint64_t ki = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  int tri = -1, cat1 = 0, cat2 = 0, callable = 0;
  bool tie_alt = false, counted = false;
  if (ki < n_keys) {
    const unsigned long long key = keys[ki];
    const uint32_t c = (uint32_t)(key >> 36);
    const int32_t pos = (int32_t)((key >> 4) & 0xffffffffull) - 1;
    const hm_chunk ch = chunks[c];
    const uint32_t n = site_n[ki], lo = site_lo[ki];
    int cnt[6] = {0, 0, 0, 0, 0, 0};
    int h0 = 0, h1 = 0;
    bool bq_zero = false;
    double S[4][3];
#pragma unroll
    for (int x = 0; x < 4; x++) { S[x][0] = 0.0; S[x][1] = 0.0; S[x][2] = 0.0; }
    for (uint32_t s = 0; s < n; s++) {
      const uint32_t e = s < n_slots ? __ldg(entries + (uint64_t)s * stride + ki)
                                     : norm_entry(b, p, ch, pair_flag[pair_off[c] + (lo + s - ch.read_lo)], lo + s, pos);
      if (e == HM_ENT_UNWRITTEN) continue; // a read of the range that does not reach the site
      const uint32_t a = e & 7u;
      cnt[4] += (int)((e >> 11) & 255u);
      if (a == HM_ENT_NONE) continue;
      if (a == 5u) { cnt[5]++; continue; }
      const int bq = (int)((e >> 3) & 255u);
      if (bq == 0) bq_zero = true;
      const double x0 = s_lut[0][bq], x1 = s_lut[1][bq], x2 = s_lut[2][bq];
#pragma unroll
      for (int x = 0; x < 4; x++) {
        if ((int)a == x) {
          cnt[x]++;
          S[x][0] = __dadd_rn(S[x][0], x0); S[x][1] = __dadd_rn(S[x][1], x1); S[x][2] = __dadd_rn(S[x][2], x2);
        }
      }
      const uint32_t hap = (e >> 19) & 3u;
      h0 += (hap == 0u); h1 += (hap == 1u);
      callable += (int)((e >> 21) & 1u);
    }
    const uint8_t rb = (pos >= 0 && (uint64_t)pos < ref_len) ? __ldg(refseq + pos) : (uint8_t)0;
    const int ridx = rb == 'A' ? 0 : rb == 'T' ? 1 : rb == 'G' ? 2 : rb == 'C' ? 3 : -1;
    counted = ridx >= 0 && callable > 0;
    if (counted) {
      if (bq_zero) s_err = HM_ERR_BQ_ZERO;
      if (p.phase && !(h0 >= p.min_hap_count && h1 >= p.min_hap_count)) cat1 = 2;
      else {
        double pl[10];
#pragma unroll
        for (int g = 0; g < 10; g++) pl[g] = gt_pl_dev(S, g, ridx, -1);
        int gq; bool tie;
        const int best = argmin_gt_dev(pl, &gq, &tie);
        const int state = gt_state_dev(c_gt_b1[best], c_gt_b2[best], ridx);
        const int depth = cnt[0] + cnt[1] + cnt[2] + cnt[3] + cnt[5];
        const int ref_count = cnt[ridx];
        if (state != 0) cat1 = state == 1 ? 3 : state == 2 ? 4 : 5;
        else {
          cat1 = 6;
          if (cnt[5] != 0 || cnt[4] != 0) cat2 = 7;
          else if ((double)depth > p.md_threshold) cat2 = 8;
          else if (depth == ref_count) {
            if (gq < p.min_gq) cat2 = 10;
            else if (ref_count < p.min_ref_count) cat2 = 9;
            else { cat2 = 13; tri = tri_bin_dev(refseq, ref_len, pos); }
          } else {
            // alts in canonical A,T,G,C order (the reference iterates a set: order flagged, not guessed)
            int alt = -1, amax = -1, nmax = 0;
#pragma unroll
            for (int x = 0; x < 4; x++) {
              if (x == ridx || cat2) continue;
              if (cnt[x] > 0) {
                const uint64_t skey = ((uint64_t)(uint32_t)(pos + 1) << 4) | ((uint64_t)ridx << 2) | (uint64_t)x;
                if (!p.non_human_sample && key_in_dev(sets.pon, sets.n_pon, skey)) cat2 = 11;
                else if (!p.non_human_sample && key_in_dev(sets.common, sets.n_common, skey)) cat2 = 12;
              }
              if (cnt[x] > amax) { amax = cnt[x]; alt = x; nmax = 1; }
              else if (cnt[x] == amax) nmax++;
            }
            if (!cat2) {
              tie_alt = nmax > 1;
#pragma unroll
              for (int g = 0; g < 10; g++) pl[g] = gt_pl_dev(S, g, ridx, alt); // get_germ_gq(alt 1-char)
              int gq2; bool tie2;
              argmin_gt_dev(pl, &gq2, &tie2);
              if (gq2 < p.min_gq) cat2 = 10;
              else if (!(ref_count >= p.min_ref_count && cnt[alt] >= p.min_alt_count)) cat2 = 9;
              else { cat2 = 13; tri = tri_bin_dev(refseq, ref_len, pos); }
            }
          }
        }
      }
    }
    if constexpr (kTrack) { if (tri >= 0) track[track_at(track_off, c, ch.start, pos)] = (uint32_t)callable; }
  }
  {
    const unsigned cv = counted ? (unsigned)callable : 0u;
#pragma unroll
    for (int i = 1; i < HM_NORM_LOG_LEN; i++) {
      const unsigned v = __reduce_add_sync(HM_FULL, (i == 1 || i == cat1 || i == cat2) ? cv : 0u);
      if (lane == 0 && v) atomicAdd(&s_log[i], (unsigned long long)v);
    }
  }
  if (tri >= 0) { atomicAdd(&s_ref[tri], 1ull); atomicAdd(&s_ccs[tri], (unsigned long long)callable); }
  if (tie_alt) atomicAdd(&s_tie, 1ull);
  __syncthreads();
  if (threadIdx.x < HM_TRI_BINS) {
    if (s_ccs[threadIdx.x]) atomicAdd(&out->ccs_tri[threadIdx.x], s_ccs[threadIdx.x]);
    if (s_ref[threadIdx.x]) atomicAdd(&out->ref_tri[threadIdx.x], s_ref[threadIdx.x]);
  }
  if (threadIdx.x < HM_NORM_LOG_LEN && s_log[threadIdx.x]) atomicAdd(&out->log[threadIdx.x], s_log[threadIdx.x]);
  if (threadIdx.x == 0) {
    if (s_tie) atomicAdd(&out->alt_tie, s_tie);
    if (s_err) out->err = s_err;
  }
}

// k_site_range for a plain key array of known length (the site list of k_norm_bits)
__global__ void __launch_bounds__(256) k_norm_site_range(DevBatch b, const hm_chunk* chunks, const unsigned long long* keys,
                                                         uint64_t n_keys, uint32_t* site_lo, uint32_t* site_n) {
  const uint64_t ki = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (ki >= n_keys) return;
  const unsigned long long key = keys[ki];
  const hm_chunk ch = chunks[(uint32_t)(key >> 36)];
  const int32_t rpos = (int32_t)((key >> 4) & 0xffffffffull) - 1;
  const uint32_t n_in = ch.read_hi - ch.read_lo;
  const uint32_t lo = count_le_kary_i32(b.pmax_tend + ch.read_lo, n_in, rpos - 1);
  const uint32_t hi = count_le_kary_i32(b.tstart + ch.read_lo, n_in, rpos);
  site_lo[ki] = ch.read_lo + lo;
  site_n[ki] = hi > lo ? hi - lo : 0u;
}

// ============================================================================ k_phase_edges
// `himut phase` edge counting (phaselib.get_edges, src/himut/phaselib.py:16-67): for every primary read with
// MAPQ >= min_mapq that covers at least two hetSNPs (hpos in (tstart, tend]), every ordered pair (a < b) of them
// whose bases both have BQ >= min_bq adds one to a 2 x 2 table: cis1 (ref, ref), cis2 (non-ref, non-ref),
// trans1 (ref, non-ref), trans2 (non-ref, ref).  Tables live in a band: counts[(a * band + (b - a - 1)) * 4 + k].
// One warp per read: lanes classify the read at its hetSNPs (32 at a time, states kept in shared memory), then
// lanes enumerate the pairs.  *need_band reports the widest pair seen so the host can retry with a wider band.
#define HM_EDGE_MAX_SNPS 1024 // hetSNPs per read held in shared memory
__global__ void __launch_bounds__(128) k_phase_edges(DevBatch b, const int32_t* hpos, const uint8_t* href, uint32_t n_snp,
                                                     int32_t min_bq, int32_t min_mapq, int32_t min_tstart, uint32_t band,
                                                     unsigned int* counts, unsigned int* need_band) {
  __shared__ uint8_t s_state[4][HM_EDGE_MAX_SNPS];
  const uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (r >= b.n_reads) return;
  if (b.flags[r] & HM_READ_SECONDARY) return;           // BAM.is_primary (bamlib.py:17-20)
  if ((int32_t)b.mapq[r] < min_mapq) return;
  const int32_t ts = b.tstart[r], te = b.tend[r];
  if (ts < min_tstart) return;                           // counted with the previous window of the contig
  const uint32_t idx = upper_bound_dev(hpos, n_snp, ts), jdx = upper_bound_dev(hpos, n_snp, te);
  if (jdx - idx < 2) return;
  const uint32_t k = jdx - idx;
  if (k > HM_EDGE_MAX_SNPS) { if (lane == 0) atomicMax(need_band, 0xffffffffu); return; }
  for (uint32_t i = lane; i < k; i += 32) {
    int bq, ins;
    const int a = read_allele_fast(b, (uint32_t)r, hpos[idx + i] - 1, ts, (int)href[idx + i], &bq, &ins);
    // tpos2qbase: deleted base ("-", 0); every covered position has an entry (cslib.py:153-170)
    uint8_t st = 2;                                      // 2: skipped (BQ below min_bq)
    if (!(bq < min_bq)) st = (a >= 0 && a < 4 && a == (int)href[idx + i]) ? 0 : 1;
    s_state[wid][i] = st;
  }
  __syncwarp();
  if (k - 1 > band) { if (lane == 0) atomicMax(need_band, k - 1); return; }
  // pairs (x, y), x < y: lane strides over y for each x
  for (uint32_t x = 0; x + 1 < k; x++) {
    const uint32_t sx = s_state[wid][x];
    if (sx == 2u) continue;
    for (uint32_t y = x + 1 + lane; y < k; y += 32) {
      const uint32_t sy = s_state[wid][y];
      if (sy == 2u) continue;
      const uint32_t kind = sx == 0u ? (sy == 0u ? 0u : 2u) : (sy == 1u ? 1u : 3u);
      atomicAdd(counts + ((uint64_t)(idx + x) * band + (y - x - 1)) * 4 + kind, 1u);
    }
  }
}

