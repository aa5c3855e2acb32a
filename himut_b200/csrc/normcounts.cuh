// normcounts.cuh — callable-base half of `himut normcounts` on sm_100a
// (normcounts.get_callable_tricounts, src/himut/normcounts.py:240-419).
//
//   k_pair_info        per (chunk, read) pair: fetch rule, [--phase] read haplotype, read gates,
//                      distinct-qname mark (normcounts.py:292-314)
//   k_norm_tiles_tma   single pass that genotypes every covered position from ordered fp64 adds,
//                      one thread per reference position of a 512-position tile (see below).  It
//                      runs where the bit-vector pass of normbits.cuh does not apply: parameters
//                      outside the certified domain, a chunk that starts below position 0, 2^32
//                      or more cal words in one batch.  Only 33+33 trinucleotide bins and 14
//                      counters leave the SM (shared-memory tallies, one global atomic per bin
//                      per CTA).
//   k_ref_tricounts    reference trinucleotide counts (reflib.get_chrom_tricount)
//
// k_norm_tiles_tma is bound by instruction issue / the fp64 pipe rather than by HBM; see DESIGN.md.
#pragma once
#include "kernels.cuh"

struct NormOut { // device tallies
  unsigned long long ccs_tri[HM_TRI_BINS];
  unsigned long long ref_tri[HM_TRI_BINS];
  unsigned long long log[HM_NORM_LOG_LEN];
  unsigned long long alt_tie;
  int err;
};

// pair_flag bits
#define HM_PF_FETCHED 1u
#define HM_PF_PASS 2u
#define HM_PF_HAP_SHIFT 2

__global__ void __launch_bounds__(256) k_pair_info(DevBatch b, DevParams p, DevPhase ph, const hm_chunk* chunks, uint32_t n_chunks,
                                                   const uint64_t* pair_off, uint64_t n_pairs, uint8_t* pair_flag,
                                                   uint8_t* qname_seen) {
  const uint64_t pr = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (pr >= n_pairs) return;
  const uint32_t c = upper_bound_dev(pair_off, n_chunks + 1, pr) - 1;
  const hm_chunk ch = chunks[c];
  const uint64_t r = (uint64_t)ch.read_lo + (pr - pair_off[c]);
  uint32_t f = 0;
  if (!(b.flags[r] & HM_READ_SECONDARY) && b.tstart[r] < ch.end && b.tend[r] > ch.start) {
    f = HM_PF_FETCHED;
    int hap = 2;
    if (p.phase) hap = warp_read_hap(b, r, ph, ch.phase_set, lane);
    f |= (uint32_t)hap << HM_PF_HAP_SHIFT;
    if ((!p.phase || hap < 2) && b.gate[r]) {
      f |= HM_PF_PASS;
      if (lane == 0) qname_seen[b.qname_id[r]] = 1;
    }
  }
  if (lane == 0) pair_flag[pr] = (uint8_t)f;
}

// normcounts.get_tri_context (normcounts.py:49-62) -> bin in mutlib.tri_lst order, 32 = other
__device__ __forceinline__ int tri_code(uint8_t ch) { return ch == 'A' ? 0 : ch == 'C' ? 1 : ch == 'G' ? 2 : ch == 'T' ? 3 : -1; }
__device__ __forceinline__ int tri_bin_dev(const uint8_t* seq, uint64_t n, int64_t pos) {
  if (pos < 1 || (uint64_t)pos + 1 >= n) return 32;
  int t0 = tri_code(seq[pos - 1]), t1 = tri_code(seq[pos]), t2 = tri_code(seq[pos + 1]);
  if (t1 == 0 || t1 == 2) { // purine centre: reverse complement
    const int u0 = t2 < 0 ? -1 : 3 - t2, u2 = t0 < 0 ? -1 : 3 - t0;
    t0 = u0; t1 = 3 - t1; t2 = u2;
  }
  if (t0 < 0 || t1 < 0 || t2 < 0) return 32;
  return t0 * 8 + (t1 == 3 ? 4 : 0) + t2;
}

// ============================================================================ k_norm_tiles_tma
// Warp-specialised and persistent.  The tile's reads are walked in file order, so each thread sees "its" column of
// the pileup in the reference's append order (6 allele counts, the ordered fp64 sums of the genotype model, the
// callable-read count of update_tri2count, normcounts.py:65-110, and the haplotype counts); then the thread genotypes
// its position and runs the filter cascade (normcounts.py:317-400).
//   producer warp: for the tile's reads, 32 at a time (one lane per read), finds the slice of the
//     op stream and of the mismatch list that touches the tile (8-ary searches), writes a compact
//     descriptor into shared memory and stages the read's quality bytes and 2-bit bases for the
//     tile with cp.async.bulk (TMA 1-D bulk copy, 16-byte granules) completing on an mbarrier;
//   16 consumer warps: one reference position per thread; they wait on the stage's "full"
//     mbarrier, walk its reads in file order out of shared memory and release the stage through
//     the "empty" mbarrier.  Per-position state lives in registers: 6 counts, the ordered fp64
//     sums of the position's first-seen allele (other alleles go to a rarely taken path), the
//     callable count and the haplotype tallies.
// A stage is one batch of <= 32 reads of one tile; the producer runs ahead across tiles.
#define HM_TW 512            // positions per tile = consumer threads
#define HM_NPROD 4           // producer warps, alternating batches
#define HM_NSTAGE 4
#define HM_SLOTS 32          // reads per stage
#define HM_BQ_BUF 640        // staged quality bytes per read: tile + insertions + alignment slack
#define HM_SEQ_BUF 176       // staged 2-bit bytes per read
#define HM_MAX_SOPS 12       // ops of one read inside one tile kept in the descriptor
#define HM_MAX_SMM 8         // mismatch-list entries near the tile the producer folds into `blocked`

// One read's view of one tile.  The producer folds everything that is not "plain matched base"
// into two 512-bit masks so the consumers' common case needs no op search:
//   special  positions that need the op list: substitutions, deleted bases, the base after an
//            insertion, and bases whose query offset differs from their 32-position chunk's
//   blocked  matched bases that update_tri2count would not count because of the trim range or
//            the mismatch window (normcounts.py:82-94)
//   wdelta   per 32-position chunk: query position = tile-relative position + wdelta
struct __align__(16) TileSlot {
  uint8_t bq[HM_BQ_BUF];
  uint8_t seq[HM_SEQ_BUF];
  uint32_t special[HM_TW / 32];
  uint32_t blocked[HM_TW / 32];
  int32_t wdelta[HM_TW / 32];
  uint32_t op_w[HM_MAX_SOPS];   // op word
  uint32_t op_t[HM_MAX_SOPS];   // reference offset from tstart
  uint32_t op_q[HM_MAX_SOPS];   // query position
  // what the consumers read: one 16-byte head per slot, one 16-byte record per 32-position chunk
  uint4 head;                   // x flags (HM_PF_* | HM_SLOT_SLOW), y cov_lo | cov_hi << 16, z q_base, w n_ops
  uint4 chunk[HM_TW / 32];      // x special, y blocked, z wdelta, w unused
  int32_t ts, te, qlen;
  uint32_t read;                // read index (slow path)
};
#define HM_SLOT_SLOW 0x100u

struct __align__(16) TileStage {
  TileSlot slot[HM_SLOTS];
  int32_t n_slots;
  int32_t last;                 // last batch of its tile
  int32_t pad[2];
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  }
}
// same, for the producer warps: sleep between probes so they do not take issue slots from the consumers
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  for (;;) {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    if (ok) break;
    __nanosleep(256);
  }
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ask for [src, src + bytes) to be brought into L2 (bytes: a multiple of 16); nothing waits for it
__device__ __forceinline__ void bulk_prefetch_l2(const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}

// set bits [lo, hi) of a 512-bit mask in shared memory (single writer)
__device__ __forceinline__ void mask_set(uint32_t* m, int32_t lo, int32_t hi) {
  if (lo < 0) lo = 0;
  if (hi > HM_TW) hi = HM_TW;
  while (lo < hi) {
    const int32_t wi = lo >> 5, b0 = lo & 31, n = min(32 - b0, hi - lo);
    m[wi] |= (n == 32 ? 0xffffffffu : ((1u << n) - 1u)) << b0;
    lo += n;
  }
}

// producer lane: descriptor + bulk copies of read r for tile [t0, t1)
__device__ __forceinline__ void fill_slot(const DevBatch& b, const DevParams& p, TileSlot* S, uint64_t* full_bar, uint32_t r,
                                          uint32_t pf, int32_t t0, int32_t t1) {
  const int32_t ts = __ldg(b.tstart + r), te = __ldg(b.tend + r);
  uint32_t flags = 0, nb_bq = 0, nb_seq = 0, cov = 1u, q_base_out = 0, n_ops_out = 0;
  const uint8_t *src_bq = nullptr, *src_seq = nullptr;
  if ((pf & HM_PF_FETCHED) && ts < t1 && te >= t0) {
    const uint32_t n = __ldg(b.n_ops + r);
    const uint64_t o0 = __ldg(b.op_off + r);
    const int32_t qlen = __ldg(b.qlen + r);
    if (n > 0) {
      flags = pf & 0xffu;
      const uint32_t reflen = (uint32_t)(te - ts);
      const uint32_t woff = (uint32_t)max(t0 - ts, 0);
      const uint32_t eoff = min((uint32_t)(t1 - 1 - ts), reflen); // last offset the tile can ask for
      uint32_t k0 = count_le_kary(b.op_t + o0, n, woff) - 1;
      while (k0 > 0 && __ldg(b.op_t + o0 + k0 - 1) == woff) k0--;
      const uint32_t k1 = count_le_kary(b.op_t + o0, n, eoff);
      const uint32_t ns = k1 - k0;
      // mismatch-list slice near the tile (window reach <= 2w, list is 1-based)
      const int32_t* mm = b.mm_pos + o0;
      const uint32_t nmm = (uint32_t)__ldg(b.n_mm + r);
      const int w = p.mismatch_window;
      const uint32_t m_lo = count_le_kary_i32(mm, nmm, t0 - 2 * w - 2);
      const uint32_t m_hi = count_le_kary_i32(mm, nmm, t1 + 2 * w + 2);
      bool slow = ns > HM_MAX_SOPS || (m_hi - m_lo) > HM_MAX_SMM;
      uint32_t q_lo = 0, q_hi = 0;
      if (!slow) {
        for (uint32_t i = 0; i < ns; i++) {
          const uint32_t wd = __ldg(b.ops + o0 + k0 + i), ot = __ldg(b.op_t + o0 + k0 + i), oq = __ldg(b.op_q + o0 + k0 + i);
          S->op_w[i] = wd; S->op_t[i] = ot; S->op_q[i] = oq;
          const uint32_t kind = wd & 3u, v = wd >> 2;
          if (i == 0) q_lo = oq + ((kind == HM_OP_MATCH && woff > ot) ? woff - ot : 0u);
          if (i == ns - 1) {
            if (kind == HM_OP_MATCH) q_hi = oq + min(v, eoff + 1 - ot);
            else q_hi = oq + (uint32_t)op_qry_len(wd);
          }
        }
        // fold ops, trim range and mismatch window into the masks
        int32_t mmv[HM_MAX_SMM];
        const uint32_t nmv = m_hi - m_lo;
        for (uint32_t i = 0; i < HM_MAX_SMM; i++) mmv[i] = i < nmv ? __ldg(mm + m_lo + i) : 0;
        for (int wi = 0; wi < HM_TW / 32; wi++) { S->special[wi] = 0; S->blocked[wi] = 0; S->wdelta[wi] = INT32_MIN; }
        const int32_t trim_s = (int32_t)floor(__dmul_rn(p.min_trim, (double)qlen));
        const int32_t trim_e = (int32_t)ceil(__dmul_rn(__dsub_rn(1.0, p.min_trim), (double)qlen));
        const int32_t W = t1 - t0;
        for (uint32_t i = 0; i < ns; i++) {
          const uint32_t wd = S->op_w[i];
          const uint32_t kind = wd & 3u;
          const int32_t a = ts + (int32_t)S->op_t[i] - t0, rl = op_ref_len(wd);
          if (kind == HM_OP_MATCH) {
            const int32_t lo_p = max(a, 0), hi_p = min(a + rl, W);
            if (lo_p >= hi_p) continue;
            const int32_t qpos0 = (int32_t)S->op_q[i], delta = qpos0 - a;
            // bamlib.get_mismatch_range anchored at the block start (normcounts.py:82)
            const int qs = qpos0 - w, qe2 = qpos0 + w;
            int u, d;
            if (qs < 0) { u = w + qs; d = w + (-qs); }
            else if (qe2 > qlen) { u = w + (qe2 - qlen); d = qlen - qpos0; }
            else { u = w; d = w; }
            if (p.max_mismatch_count == 0) {
              for (uint32_t m = 0; m < nmv; m++) mask_set(S->blocked, max(mmv[m] - d - t0, lo_p), min(mmv[m] + u - t0 + 1, hi_p));
            } else {
              // general threshold: count per position (rare setting; window reach is small)
              for (int32_t pp = lo_p; pp < hi_p; pp++) {
                int mc = 0;
                for (uint32_t m = 0; m < nmv; m++) mc += (mmv[m] >= t0 + pp - u && mmv[m] <= t0 + pp + d);
                if (mc > p.max_mismatch_count) mask_set(S->blocked, pp, pp + 1);
              }
            }
            mask_set(S->blocked, lo_p, min(hi_p, trim_s - delta));          // q < trim_s
            mask_set(S->blocked, max(lo_p, trim_e - delta + 1), hi_p);      // q > trim_e
            for (int32_t cidx = lo_p >> 5; cidx <= (hi_p - 1) >> 5; cidx++) {
              if (S->wdelta[cidx] == INT32_MIN) S->wdelta[cidx] = delta;
              else if (S->wdelta[cidx] != delta) mask_set(S->special, max(lo_p, cidx * 32), min(hi_p, cidx * 32 + 32));
            }
          } else if (kind == HM_OP_DEL) {
            mask_set(S->special, max(a, 0), min(a + rl, W));
          } else if (a >= 0 && a < W) {
            mask_set(S->special, a, a + 1); // substitution, or the base an insertion precedes
          }
        }
        cov = (uint32_t)max(ts - t0, 0) | ((uint32_t)max(min(te - 1 - t0, W - 1), 0) << 16);
        if (te - 1 < t0) cov = 1u; // lo 1 > hi 0: nothing aligned inside the tile (trailing insertion only)
        const uint32_t qb = q_lo & ~63u;
        const uint32_t qe = min((q_hi + 15u) & ~15u, ((uint32_t)qlen + 15u) & ~15u);
        const uint32_t sb0 = qb >> 2, sb1 = min(((((q_hi + 3u) >> 2) + 15u) & ~15u), (((((uint32_t)qlen + 3u) >> 2) + 15u) & ~15u));
        q_base_out = qb;
        if (q_hi > q_lo) {
          if (qe - qb > HM_BQ_BUF || sb1 - sb0 > HM_SEQ_BUF) slow = true;
          else { nb_bq = qe - qb; nb_seq = sb1 - sb0; src_bq = b.bq + __ldg(b.bq_off + r) + qb; src_seq = b.seq + __ldg(b.seq_off + r) + sb0; }
        }
      }
      if (slow) { flags |= HM_SLOT_SLOW; nb_bq = nb_seq = 0; }
      n_ops_out = slow ? 0 : ns;
      S->ts = ts; S->te = te; S->qlen = qlen; S->read = r;
      if (!slow)
        for (int wi = 0; wi < HM_TW / 32; wi++) S->chunk[wi] = make_uint4(S->special[wi], S->blocked[wi], (uint32_t)S->wdelta[wi], 0u);
    }
  }
  S->head = make_uint4(flags, cov, q_base_out, n_ops_out);
  // the descriptor is complete: arrive (release) last, then let the bulk copies land on the barrier
  if (nb_bq + nb_seq == 0) mbar_arrive(full_bar);
  else {
    mbar_arrive_expect_tx(full_bar, nb_bq + nb_seq);
    bulk_g2s(S->bq, src_bq, nb_bq, full_bar);
    bulk_g2s(S->seq, src_seq, nb_seq, full_bar);
  }
}

// tri_bin_dev with the three bases already in registers
__device__ __forceinline__ int tri_bin3(uint8_t l, uint8_t m, uint8_t r, int64_t pos, uint64_t n) {
  if (pos < 1 || (uint64_t)pos + 1 >= n) return 32;
  int t0 = tri_code(l), t1 = tri_code(m), t2 = tri_code(r);
  if (t1 == 0 || t1 == 2) {
    const int u0 = t2 < 0 ? -1 : 3 - t2, u2 = t0 < 0 ? -1 : 3 - t0;
    t0 = u0; t1 = 3 - t1; t2 = u2;
  }
  if (t0 < 0 || t1 < 0 || t2 < 0) return 32;
  return t0 * 8 + (t1 == 3 ? 4 : 0) + t2;
}

__global__ void __launch_bounds__(HM_TW + 32 * HM_NPROD, 1) k_norm_tiles_tma(DevBatch b, DevParams p, DevSets sets, DevLut lut, const hm_chunk* chunks,
                                                                   uint32_t n_chunks, const uint64_t* pair_off, const uint8_t* pair_flag,
                                                                   const uint64_t* tile_off, uint32_t n_tiles, const uint8_t* refseq,
                                                                   uint64_t ref_len, NormOut* out) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  TileStage* stages = reinterpret_cast<TileStage*>(smem_raw);
  __shared__ double s_lut[3][256];
  __shared__ uint64_t full_bar[HM_NSTAGE], empty_bar[HM_NSTAGE];
  __shared__ unsigned long long s_ccs[HM_TRI_BINS], s_ref[HM_TRI_BINS], s_log[HM_NORM_LOG_LEN], s_tie;
  __shared__ unsigned int s_wccs[HM_TW / 32][HM_TRI_BINS + 1], s_wref[HM_TW / 32][HM_TRI_BINS + 1]; // per-warp bins
  __shared__ int s_err;
  const int tid = threadIdx.x, lane = tid & 31;
  const bool is_producer = tid >= HM_TW;
  for (int i = tid; i < (HM_TW / 32) * (HM_TRI_BINS + 1); i += blockDim.x) { (&s_wccs[0][0])[i] = 0; (&s_wref[0][0])[i] = 0; }
  for (int i = tid; i < 768; i += blockDim.x) s_lut[i >> 8][i & 255] = __ldg(lut.lut + i);
  if (tid < HM_TRI_BINS) { s_ccs[tid] = 0; s_ref[tid] = 0; }
  if (tid < HM_NORM_LOG_LEN) s_log[tid] = 0;
  if (tid == 0) {
    s_tie = 0; s_err = 0;
    for (int i = 0; i < HM_NSTAGE; i++) { mbar_init(&full_bar[i], HM_SLOTS); mbar_init(&empty_bar[i], HM_TW / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  uint32_t batch_no = 0; // same sequence on both sides
  if (is_producer) {
    // ------------------------------------------------------------------ producer warps
    const uint32_t pw = (uint32_t)(tid - HM_TW) >> 5;
    uint32_t c = 0; // tiles are visited in increasing order: a running chunk cursor replaces a search
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      while (c + 1 < n_chunks && (uint64_t)tile >= __ldg(tile_off + c + 1)) c++;
      const hm_chunk ch = chunks[c];
      const int32_t t0 = ch.start + (int32_t)(tile - tile_off[c]) * HM_TW;
      const int32_t t1 = min(t0 + HM_TW, ch.end);
      const uint32_t n_in = ch.read_hi - ch.read_lo;
      const uint32_t r_lo = ch.read_lo + warp_count_below<true>(b.pmax_tend + ch.read_lo, n_in, t0, lane);
      const uint32_t r_hi = ch.read_lo + warp_count_below<true>(b.tstart + ch.read_lo, n_in, t1, lane);
      const uint64_t pbase = pair_off[c];
      uint32_t r0 = r_lo;
      do {
        if (batch_no % HM_NPROD != pw) { batch_no++; r0 += HM_SLOTS; continue; }
        const uint32_t st = batch_no % HM_NSTAGE, ph = (batch_no / HM_NSTAGE) & 1;
        mbar_wait_backoff(&empty_bar[st], ph ^ 1);
        TileStage* T = &stages[st];
        const uint32_t r = r0 + lane;
        const uint32_t nb = min(r_hi > r0 ? r_hi - r0 : 0u, (uint32_t)HM_SLOTS);
        if (lane == 0) { T->n_slots = (int32_t)nb; T->last = (r0 + HM_SLOTS >= r_hi) ? 1 : 0; }
        if ((uint32_t)lane < nb) {
          const uint32_t pf = pair_flag[pbase + (r - ch.read_lo)];
          fill_slot(b, p, &T->slot[lane], &full_bar[st], r, pf, t0, t1);
        } else {
          mbar_arrive(&full_bar[st]);
        }
        batch_no++;
        r0 += HM_SLOTS;
      } while (r0 < r_hi);
    }
    return;
  }

  // -------------------------------------------------------------------- consumer warps
  const int w = p.mismatch_window;
  uint32_t c = 0;
  for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    while (c + 1 < n_chunks && (uint64_t)tile >= __ldg(tile_off + c + 1)) c++;
    const hm_chunk ch = chunks[c];
    const int32_t t0 = ch.start + (int32_t)(tile - tile_off[c]) * HM_TW;
    const int32_t t1 = min(t0 + HM_TW, ch.end);
    const int32_t pos = t0 + tid;
    const bool live = pos < t1 && pos >= 0 && (uint64_t)pos < ref_len;
    // reference bases of the position and its neighbours now, so the loads hide behind the read loop
    const uint8_t rb = live ? __ldg(refseq + pos) : (uint8_t)0;
    const uint8_t rb_l = (live && pos >= 1) ? __ldg(refseq + pos - 1) : (uint8_t)0;
    const uint8_t rb_r = (live && (uint64_t)pos + 1 < ref_len) ? __ldg(refseq + pos + 1) : (uint8_t)0;
    const int wbase = tid & ~31; // first tile-relative position of this warp

    int n_main = 0, n_oth[3] = {0, 0, 0}, cnt_ins = 0, cnt_del = 0;
    int a_main = -1;
    double M0 = 0.0, M1 = 0.0, M2 = 0.0;             // ordered sums of the first-seen allele
    double O[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}}; // alleles (a_main + 1..3) & 3
    int callable = 0, h0 = 0, h1 = 0;
    bool bq_zero = false;

    for (;;) {
      const uint32_t st = batch_no % HM_NSTAGE, ph = (batch_no / HM_NSTAGE) & 1;
      mbar_wait(&full_bar[st], ph);
      const TileStage* T = &stages[st];
      const int nslots = T->n_slots;
      const int last = T->last;
      for (int si = 0; si < nslots; si++) {
        const TileSlot* S = &T->slot[si];
        const uint4 hd = S->head;                       // one broadcast LDS.128
        const uint32_t fl = hd.x;
        if (!(fl & HM_PF_FETCHED)) continue;            // uniform
        int a = -1, bq = 0, ins = 0;
        bool count_it = false; // callable by update_tri2count (normcounts.py:65-110)
        if (!(fl & HM_SLOT_SLOW)) {
          const uint4 ci = S->chunk[tid >> 5];          // one broadcast LDS.128
          const int cov_lo = (int)(hd.y & 0xffffu), cov_hi = (int)(hd.y >> 16);
          const bool special = (ci.x >> lane) & 1u;
          if (ci.x == 0u && (wbase > cov_hi || wbase + 31 < cov_lo)) continue; // uniform: chunk not covered
          if (!special) {
            // plain matched base: query position from the chunk's offset, data from the staged bytes
            if (tid >= cov_lo && tid <= cov_hi) {
              const uint32_t q = (uint32_t)(tid + (int32_t)ci.z);
              bq = S->bq[q - hd.z];
              a = (S->seq[(q >> 2) - (hd.z >> 2)] >> (2 * (q & 3u))) & 3;
              count_it = !((ci.y >> lane) & 1u) && bq >= p.min_bq;
            }
          } else {
            // substitution / deleted base / base after an insertion / odd query offset: op list
            const int32_t ts = S->ts;
            if (pos >= ts && pos <= S->te) {
              const uint32_t off = (uint32_t)(pos - ts);
              const uint32_t n = hd.w;
              uint32_t k = 0, wd = S->op_w[0], t_op = S->op_t[0];
              for (;;) {
                if (t_op == off && (wd & 3u) == HM_OP_INS) ins++;
                if (k + 1 >= n) break;
                const uint32_t tn = S->op_t[k + 1];
                if (tn > off) break;
                k++; wd = S->op_w[k]; t_op = tn;
              }
              const uint32_t kind = wd & 3u;
              const uint32_t rl = (uint32_t)op_ref_len(wd);
              if (rl != 0 && off >= t_op && off < t_op + rl) {
                if (kind == HM_OP_DEL) a = 5;
                else {
                  const uint32_t q = S->op_q[k] + (kind == HM_OP_MATCH ? off - t_op : 0u);
                  bq = S->bq[q - hd.z];
                  a = kind == HM_OP_SUB ? (int)((wd >> 5) & 3u) : (int)((S->seq[(q >> 2) - (hd.z >> 2)] >> (2 * (q & 3u))) & 3u);
                  count_it = kind == HM_OP_SUB || (!((ci.y >> lane) & 1u) && bq >= p.min_bq);
                }
              }
            }
          }
        } else {
          // pathological read (many ops / long insertions inside one tile): global-memory lookups
          const int32_t ts = S->ts;
          if (live && pos >= ts && pos <= S->te) {
            const uint32_t off = (uint32_t)(pos - ts);
            const uint32_t r = S->read;
            const uint32_t n = __ldg(b.n_ops + r);
            const uint64_t o0 = __ldg(b.op_off + r);
            const int k = (int)count_le_kary(b.op_t + o0, n, off) - 1;
            for (int j = k; j >= 0 && __ldg(b.op_t + o0 + j) == off; j--)
              if ((__ldg(b.ops + o0 + j) & 3u) == HM_OP_INS) ins++;
            const uint32_t wd = __ldg(b.ops + o0 + k);
            const uint32_t kind = wd & 3u, t_op = __ldg(b.op_t + o0 + k), q0 = __ldg(b.op_q + o0 + k);
            const uint32_t rl = (uint32_t)op_ref_len(wd);
            if (rl != 0 && off < t_op + rl) {
              if (kind == HM_OP_DEL) a = 5;
              else {
                const uint32_t q = q0 + (kind == HM_OP_MATCH ? off - t_op : 0u);
                bq = b.bq[__ldg(b.bq_off + r) + q];
                a = kind == HM_OP_SUB ? (int)((wd >> 5) & 3u) : (int)((b.seq[__ldg(b.seq_off + r) + (q >> 2)] >> (2 * (q & 3u))) & 3u);
                if (kind == HM_OP_SUB) count_it = true;
                else if (bq >= p.min_bq) {
                  const int32_t qlen = S->qlen;
                  const int32_t trim_s = (int32_t)floor(__dmul_rn(p.min_trim, (double)qlen));
                  const int32_t trim_e = (int32_t)ceil(__dmul_rn(__dsub_rn(1.0, p.min_trim), (double)qlen));
                  if (!((int32_t)q < trim_s || (int32_t)q > trim_e)) {
                    const int32_t qpos0 = (int32_t)q0;
                    const int qs = qpos0 - w, qe = qpos0 + w;
                    int u, d;
                    if (qs < 0) { u = w + qs; d = w + (-qs); }
                    else if (qe > qlen) { u = w + (qe - qlen); d = qlen - qpos0; }
                    else { u = w; d = w; }
                    const int32_t* mm = b.mm_pos + o0;
                    const uint32_t nmm = (uint32_t)__ldg(b.n_mm + r);
                    const int mc = (int)count_le_kary_i32(mm, nmm, pos + d) - (int)count_le_kary_i32(mm, nmm, pos - u - 1);
                    count_it = !(mc > p.max_mismatch_count);
                  }
                }
              }
            }
          }
        }
        cnt_ins += ins;
        cnt_del += (a == 5);
        if (a >= 0 && a < 4) {
          bq_zero |= (bq == 0);
          const double x0 = s_lut[0][bq], x1 = s_lut[1][bq], x2 = s_lut[2][bq];
          if (a_main < 0) a_main = a;
          if (a == a_main) { n_main++; M0 = __dadd_rn(M0, x0); M1 = __dadd_rn(M1, x1); M2 = __dadd_rn(M2, x2); }
          else {
            const int j = ((a - a_main) & 3) - 1;
#pragma unroll
            for (int jj = 0; jj < 3; jj++)
              if (j == jj) { n_oth[jj]++; O[jj][0] = __dadd_rn(O[jj][0], x0); O[jj][1] = __dadd_rn(O[jj][1], x1); O[jj][2] = __dadd_rn(O[jj][2], x2); }
          }
          if (p.phase) {
            const int hap = (int)(fl >> HM_PF_HAP_SHIFT) & 3;
            h0 += (hap == 0); h1 += (hap == 1);
          }
          callable += (count_it && (fl & HM_PF_PASS)) ? 1 : 0;
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[st]);
      batch_no++;
      if (last) break;
    }

    // ---- position loop body (normcounts.py:317-400) ----
    // every counted position adds its callable count to log[1] and to exactly one more counter
    // (cat1 in 2..6); homref positions (cat1 == 6) to one of 7..13 as well (cat2)
    int tri = -1, cat1 = 0, cat2 = 0;
    bool tie_alt = false;
    const int ridx = live ? (rb == 'A' ? 0 : rb == 'T' ? 1 : rb == 'G' ? 2 : rb == 'C' ? 3 : -1) : -1;
    const bool counted = ridx >= 0 && callable > 0;
    if (counted) {
      if (bq_zero) s_err = HM_ERR_BQ_ZERO;
      if (p.phase && !(h0 >= p.min_hap_count && h1 >= p.min_hap_count)) cat1 = 2;
      else if (a_main == ridx && (n_oth[0] | n_oth[1] | n_oth[2]) == 0) {
        // only the reference allele was seen: every other allele's sums are exact zeros, so the ten
        // PL collapse to four values (x + 0.0 == x): hom of it, het with it, hom / het of others
        const double p_rr = __dmul_rn(-10.0, __dadd_rn(M0, c_tab.log10_prior[0]));
        const double p_het = __dmul_rn(-10.0, __dadd_rn(M1, c_tab.log10_prior[1]));
        const double p_hetalt = __dmul_rn(-10.0, __dadd_rn(M2, c_tab.log10_prior[2]));
        const double p_homalt = __dmul_rn(-10.0, __dadd_rn(M2, c_tab.log10_prior[3]));
        double pl[10];
#pragma unroll
        for (int g = 0; g < 10; g++) {
          const int b1 = c_gt_b1[g], b2 = c_gt_b2[g];
          pl[g] = (b1 == b2) ? (b1 == ridx ? p_rr : p_homalt) : ((b1 == ridx || b2 == ridx) ? p_het : p_hetalt);
        }
        int gq; bool tie;
        const int best = argmin_gt_dev(pl, &gq, &tie);
        const int state = gt_state_dev(c_gt_b1[best], c_gt_b2[best], ridx);
        if (state != 0) cat1 = state == 1 ? 3 : state == 2 ? 4 : 5;
        else {
          cat1 = 6;
          if (cnt_del != 0 || cnt_ins != 0) cat2 = 7;
          else if ((double)n_main > p.md_threshold) cat2 = 8;
          else if (gq < p.min_gq) cat2 = 10;
          else if (n_main < p.min_ref_count) cat2 = 9;
          else { cat2 = 13; tri = tri_bin3(rb_l, rb, rb_r, pos, ref_len); }
        }
      } else {
        // rebuild S[allele][kind] and the counts from the first-seen allele's registers and the others
        double S[4][3];
        int cnt[6] = {0, 0, 0, 0, cnt_ins, cnt_del};
#pragma unroll
        for (int x = 0; x < 4; x++) {
          const int j = a_main < 0 ? -2 : ((x - a_main) & 3) - 1; // -1: main allele
          cnt[x] = j == -1 ? n_main : j == 0 ? n_oth[0] : j == 1 ? n_oth[1] : j == 2 ? n_oth[2] : 0;
#pragma unroll
          for (int k = 0; k < 3; k++) {
            double v = 0.0;
            if (j == -1) v = k == 0 ? M0 : k == 1 ? M1 : M2;
            else if (j == 0) v = O[0][k];
            else if (j == 1) v = O[1][k];
            else if (j == 2) v = O[2][k];
            S[x][k] = v;
          }
        }
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
            else { cat2 = 13; tri = tri_bin3(rb_l, rb, rb_r, pos, ref_len); }
          } else {
            // alts in canonical A,T,G,C order (the reference iterates a set: order flagged, not guessed)
            int alt = -1, amax = -1, nmax = 0;
#pragma unroll
            for (int x = 0; x < 4; x++) {
              if (x == ridx || cat2) continue;
              if (cnt[x] > 0) {
                const uint64_t key = ((uint64_t)(uint32_t)(pos + 1) << 4) | ((uint64_t)ridx << 2) | (uint64_t)x;
                if (!p.non_human_sample && key_in_dev(sets.pon, sets.n_pon, key)) cat2 = 11;
                else if (!p.non_human_sample && key_in_dev(sets.common, sets.n_common, key)) cat2 = 12;
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
              else { cat2 = 13; tri = tri_bin3(rb_l, rb, rb_r, pos, ref_len); }
            }
          }
        }
      }
    }
    // warp tallies: one REDUX per counter, lane 0 adds to the CTA's shared counters
    {
      const unsigned cv = counted ? (unsigned)callable : 0u;
#pragma unroll
      for (int i = 1; i < HM_NORM_LOG_LEN; i++) {
        const unsigned v = __reduce_add_sync(HM_FULL, (i == 1 || i == cat1 || i == cat2) ? cv : 0u);
        if (lane == 0 && v) atomicAdd(&s_log[i], (unsigned long long)v);
      }
    }
    if (tri >= 0) { atomicAdd(&s_wref[tid >> 5][tri], 1u); atomicAdd(&s_wccs[tid >> 5][tri], (unsigned)callable); }
    if (tie_alt) atomicAdd(&s_tie, 1ull);
    // move the warp's 32-bit bins into the CTA's 64-bit ones before they can overflow
    __syncwarp();
    if (lane < HM_TRI_BINS - 1 + 1 && s_wccs[tid >> 5][lane] > 0x40000000u) {
      atomicAdd(&s_ccs[lane], (unsigned long long)atomicExch(&s_wccs[tid >> 5][lane], 0u));
      atomicAdd(&s_ref[lane], (unsigned long long)atomicExch(&s_wref[tid >> 5][lane], 0u));
    }
    if (lane == 0 && s_wccs[tid >> 5][32] > 0x40000000u) {
      atomicAdd(&s_ccs[32], (unsigned long long)atomicExch(&s_wccs[tid >> 5][32], 0u));
      atomicAdd(&s_ref[32], (unsigned long long)atomicExch(&s_wref[tid >> 5][32], 0u));
    }
  }
  // fold the per-warp bins
  for (int i = lane; i < HM_TRI_BINS; i += 32) {
    if (s_wccs[tid >> 5][i]) atomicAdd(&s_ccs[i], (unsigned long long)s_wccs[tid >> 5][i]);
    if (s_wref[tid >> 5][i]) atomicAdd(&s_ref[i], (unsigned long long)s_wref[tid >> 5][i]);
  }
  // consumers only: named barrier over the 512 consumer threads, then flush the CTA tallies
  asm volatile("bar.sync 1, %0;" ::"n"(HM_TW));
  if (tid < HM_TRI_BINS) {
    if (s_ccs[tid]) atomicAdd(&out->ccs_tri[tid], s_ccs[tid]);
    if (s_ref[tid]) atomicAdd(&out->ref_tri[tid], s_ref[tid]);
  }
  if (tid < HM_NORM_LOG_LEN && s_log[tid]) atomicAdd(&out->log[tid], s_log[tid]);
  if (tid == 0) {
    if (s_tie) atomicAdd(&out->alt_tie, s_tie);
    if (s_err) out->err = s_err;
  }
}

// ============================================================================ k_ref_tricounts
// reflib.get_chrom_tricount (src/himut/reflib.py:11-33): for i in range(len(seq) - 2), skip when
// seq[i] == "N" (the *first* base of the window), otherwise count the pyrimidine-centred
// trinucleotide seq[i:i+3] (reverse complement when the centre is A/G; anything that is not
// upper-case A/C/G/T makes a key outside mutlib.tri_lst, tallied in bin 32).
// Streaming histogram: 16 windows per thread from one 16-byte load + 2 halo bytes, per-warp bins.
__global__ void __launch_bounds__(256) k_ref_tricounts(const uint8_t* seq, uint64_t n, unsigned long long* out) {
  __shared__ unsigned int s_bins[8][HM_TRI_BINS + 1];
  for (int i = threadIdx.x; i < 8 * (HM_TRI_BINS + 1); i += blockDim.x) (&s_bins[0][0])[i] = 0;
  __syncthreads();
  unsigned int* bins = s_bins[threadIdx.x >> 5];
  const uint64_t n_win = n >= 2 ? n - 2 : 0;
  for (uint64_t base = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16; base < n_win; base += (uint64_t)gridDim.x * blockDim.x * 16) {
    uint8_t c[18];
    if (base + 18 <= n && ((uintptr_t)(seq + base) & 15) == 0) {
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(seq + base));
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 16; k++) c[k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
      c[16] = __ldg(seq + base + 16); c[17] = __ldg(seq + base + 17);
    } else {
#pragma unroll
      for (int k = 0; k < 18; k++) c[k] = base + k < n ? __ldg(seq + base + k) : (uint8_t)0;
    }
#pragma unroll
    for (int k = 0; k < 16; k++) {
      if (base + k >= n_win || c[k] == 'N') continue;
      int t0 = tri_code(c[k]), t1 = tri_code(c[k + 1]), t2 = tri_code(c[k + 2]);
      if (t1 == 0 || t1 == 2) { const int u0 = t2 < 0 ? -1 : 3 - t2, u2 = t0 < 0 ? -1 : 3 - t0; t0 = u0; t1 = 3 - t1; t2 = u2; }
      const int bin = (t0 < 0 || t1 < 0 || t2 < 0) ? 32 : t0 * 8 + (t1 == 3 ? 4 : 0) + t2;
      atomicAdd(&bins[bin], 1u);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < HM_TRI_BINS; i += blockDim.x) {
    unsigned long long t = 0;
#pragma unroll
    for (int wv = 0; wv < 8; wv++) t += s_bins[wv][i];
    if (t) atomicAdd(out + i, t);
  }
}

struct hm_ctx;
static int hm_normcounts_impl(hm_ctx* ctx, const uint8_t* refseq, size_t ref_len, const hm_chunk* chunks, size_t n_chunks,
                              int64_t* ccs_tri, int64_t* ref_tri, int64_t* log, int64_t* n_alt_tie);
