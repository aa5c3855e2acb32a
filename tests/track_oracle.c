/* Test infrastructure: the callable-base track of `himut normcounts` on the CPU, for the tests of
 * HM_OPT_CALLABLE_TRACK (hm_last_callable_runs, include/himut_b200.h).
 *
 * The oracle (oracle/himut_oracle.c) is compiled in as it is, and trk_normcounts_chunks_track below is its
 * orc_normcounts_chunks_seen with one line added to the position loop: each position it counts into the tallies is
 * appended to the track (track_add).  Everything else is the oracle's text, so the tallies it returns must be the
 * oracle's; tests/test_callable_track.py checks that on every case it runs.  A runs buffer shorter than the track:
 * the first runs_cap runs are written, *n_runs says how many there are, HM_ERR_CAPACITY (the tallies are complete).
 * Built by tests/track_oracle.py with the oracle's flags. */
#include "../oracle/himut_oracle.c"

/* counted positions appended in loop order, joined into runs of one chunk and one value; n counts every run, the
 * first cap are stored */
typedef struct {
  hm_callable_run* out;
  size_t cap, n;
  hm_callable_run last;
} track_t;

static void track_add(track_t* t, uint32_t chunk, int64_t pos, uint32_t value) {
  if (t->n && t->last.chunk == chunk && (int64_t)t->last.end == pos && t->last.value == value) {
    t->last.end++;
    if (t->n <= t->cap) t->out[t->n - 1].end++;
    return;
  }
  t->last.chunk = chunk; t->last.start = (int32_t)pos; t->last.end = (int32_t)(pos + 1); t->last.value = value;
  if (t->n < t->cap) t->out[t->n] = t->last;
  t->n++;
}

int trk_normcounts_chunks_track(const hm_params* p, const hm_read_batch* b, const uint8_t* refseq,
                                size_t ref_len, const hm_chunk* chunks, size_t n_chunks,
                                const uint64_t* common, size_t n_common, const uint64_t* pon,
                                size_t n_pon, const orc_phase* ph, const uint8_t* alt_order,
                                int64_t ccs_tri[HM_TRI_BINS], int64_t ref_tri[HM_TRI_BINS],
                                int64_t log[HM_NORM_LOG_LEN], int64_t* n_alt_tie, uint8_t* qseen, size_t qseen_cap,
                                hm_callable_run* runs, size_t runs_cap, size_t* n_runs) {
  track_t track = {runs, runs ? runs_cap : 0, 0, {0, 0, 0, 0}};
  int rc = HM_OK, bq_zero = 0;
  int64_t ties = 0;
  memset(ccs_tri, 0, sizeof(int64_t) * HM_TRI_BINS);
  memset(ref_tri, 0, sizeof(int64_t) * HM_TRI_BINS);
  memset(log, 0, sizeof(int64_t) * HM_NORM_LOG_LEN);
  uint32_t max_qid = 0;
  size_t max_fetch = 1;
  for (uint64_t r = 0; r < b->n_reads; r++) if (b->qname_id[r] > max_qid) max_qid = b->qname_id[r];
  for (size_t c = 0; c < n_chunks; c++)
    if (chunks[c].read_hi > chunks[c].read_lo && (size_t)(chunks[c].read_hi - chunks[c].read_lo) > max_fetch)
      max_fetch = chunks[c].read_hi - chunks[c].read_lo;
  bitset_t seen;
  if (bitset_init(&seen, (size_t)max_qid + 1)) return HM_ERR_ARG;
  uint64_t* F = (uint64_t*)malloc(max_fetch * sizeof(uint64_t));
  uint8_t* hap = (uint8_t*)malloc(b->n_reads + 1);
  int32_t* mm = NULL; size_t mm_cap = 0;
  if (!F || !hap) { rc = HM_ERR_ARG; goto done; }

  for (size_t ci = 0; ci < n_chunks; ci++) {
    const hm_chunk* c = &chunks[ci];
    size_t nF = fetch_reads(b, c, F), nP = 0;
    for (size_t i = 0; i < nF; i++) if (!(b->flags[F[i]] & HM_READ_SECONDARY)) F[nP++] = F[i];
    nF = nP;
    pile_t P;
    if (pile_build(&P, b, F, nF)) { pile_free(&P); rc = HM_ERR_ARG; goto done; }
    size_t W = nF ? (size_t)(P.hi - P.lo) : 0;
    int32_t* callable = (int32_t*)calloc(W + 1, sizeof(int32_t)); /* rpos2count */
    int32_t* hapcnt = p->phase ? (int32_t*)calloc(W * 2 + 2, sizeof(int32_t)) : NULL; /* rpos2hap2count["0"/"1"] */
    if (!callable || (p->phase && !hapcnt)) { free(callable); free(hapcnt); pile_free(&P); rc = HM_ERR_ARG; goto done; }
    for (size_t i = 0; i < nF; i++) {
      uint64_t r = F[i];
      const uint32_t* ops = b->ops + b->op_off[r];
      uint32_t nops = b->n_ops[r];
      if (p->phase) {
        hap[r] = (uint8_t)ccs_hap(b, r, ph, c->phase_set);
        if (hap[r] < 2) { /* update_phased_allelecounts: hap counts on match / sub positions */
          int tpos = b->tstart[r];
          for (uint32_t k = 0; k < nops; k++) {
            op_t o = decode_op(ops[k]);
            if (o.kind == HM_OP_MATCH || o.kind == HM_OP_SUB)
              for (int j = 0; j < o.ref_len; j++) hapcnt[(size_t)(tpos + j - P.lo) * 2 + hap[r]]++;
            tpos += o.ref_len;
          }
        }
        if (hap[r] > 1) continue;
      }
      if (!read_passes(p, b, r)) continue;
      if (!bitset_get(&seen, b->qname_id[r])) { log[0]++; bitset_set(&seen, b->qname_id[r]); }
      /* update_tri2count (normcounts.py:65-110) */
      if (nops > mm_cap) { mm_cap = nops * 2 + 64; mm = (int32_t*)realloc(mm, mm_cap * sizeof(int32_t)); if (!mm) { free(callable); free(hapcnt); pile_free(&P); rc = HM_ERR_ARG; goto done; } }
      int nmm = 0, rpos = b->tstart[r], qpos = b->qstart[r];
      for (uint32_t k = 0; k < nops; k++) {
        op_t o = decode_op(ops[k]);
        if ((o.kind == HM_OP_SUB && o.ref != (int)HM_BASE_N) || o.kind == HM_OP_INS || o.kind == HM_OP_DEL) mm[nmm++] = rpos + 1;
        rpos += o.ref_len; qpos += o.alt_len;
      }
      double ts, te;
      trimmed_range(b->qlen[r], p->min_trim, &ts, &te);
      rpos = b->tstart[r]; qpos = b->qstart[r];
      for (uint32_t k = 0; k < nops; k++) {
        op_t o = decode_op(ops[k]);
        if (o.kind == HM_OP_MATCH) {
          int lo, hi;
          mismatch_range(rpos, qpos, b->qlen[r], p->mismatch_window, &lo, &hi);
          for (int j = 0; j < o.ref_len; j++) {
            int cnt = bisect_right_i32(mm, nmm, hi + j) - bisect_left_i32(mm, nmm, lo + j);
            if (read_bq(b, r, qpos + j) < p->min_bq) continue;
            if (cnt > p->max_mismatch_count) continue;
            if (is_trimmed(qpos + j, ts, te)) continue;
            callable[rpos + j - P.lo]++;
          }
        } else if (o.kind == HM_OP_SUB) {
          callable[rpos - P.lo]++;
        }
        rpos += o.ref_len; qpos += o.alt_len;
      }
    }
    /* position loop (normcounts.py:317-400) */
    for (int64_t rpos = c->start; rpos < c->end; rpos++) {
      if (rpos < 0 || (size_t)rpos >= ref_len) continue;
      int ridx = ascii2code(refseq[rpos]);
      if (ridx < 0) continue;
      if (!nF || rpos < P.lo || rpos >= P.hi) continue;
      int64_t tri_sum = callable[rpos - P.lo];
      if (tri_sum == 0) continue;
      log[1] += tri_sum;
      if (p->phase) {
        int h0 = hapcnt[(size_t)(rpos - P.lo) * 2], h1 = hapcnt[(size_t)(rpos - P.lo) * 2 + 1];
        if (!(h0 >= p->min_hap_count && h1 >= p->min_hap_count)) { log[2] += tri_sum; continue; }
      }
      bqlists_t L; int32_t cnt[6];
      pile_lists(&P, (int32_t)rpos, &L, cnt);
      int ins = cnt[4], del = cnt[5];
      int depth = cnt[0] + cnt[1] + cnt[2] + cnt[3] + cnt[5];
      double pl[10];
      bq_zero |= gt_pl(p, &L, ridx, -1, pl);
      int gq, tie;
      int best = argmin_gt(pl, &gq, &tie);
      int state = gt_state(GT_B1[best], GT_B2[best], ridx);
      if (state == ST_HET) { log[3] += tri_sum; continue; }
      if (state == ST_HETALT) { log[4] += tri_sum; continue; }
      if (state == ST_HOMALT) { log[5] += tri_sum; continue; }
      log[6] += tri_sum;
      if (del != 0 || ins != 0) { log[7] += tri_sum; continue; }
      if ((double)depth > p->md_threshold) { log[8] += tri_sum; continue; }
      int ref_count = cnt[ridx];
      int tri = tri_bin(refseq, ref_len, rpos);
      if (depth == ref_count) {
        if (gq < p->min_gq) { log[10] += tri_sum; continue; }
        if (ref_count < p->min_ref_count) { log[9] += tri_sum; continue; }
      } else {
        int order[3], no = 0, filtered = 0;
        if (alt_order) for (int k = 0; k < 3; k++) order[no++] = alt_order[ridx * 3 + k];
        else for (int a = 0; a < 4; a++) if (a != ridx) order[no++] = a;
        int n_hit_kinds = 0;
        for (int k = 0; k < 3 && !filtered; k++) {
          int alt = order[k];
          if (cnt[alt] == 0) continue;
          uint64_t key = site_key((int32_t)rpos + 1, ridx, alt);
          if (!p->non_human_sample && key_in(pon, n_pon, key)) { log[11] += tri_sum; filtered = 1; }
          else if (!p->non_human_sample && key_in(common, n_common, key)) { log[12] += tri_sum; filtered = 1; }
        }
        (void)n_hit_kinds;
        if (filtered) continue;
        int alt = order[0], nmax = 1;
        for (int k = 1; k < 3; k++) {
          if (cnt[order[k]] > cnt[alt]) { alt = order[k]; nmax = 1; }
          else if (cnt[order[k]] == cnt[alt]) nmax++;
        }
        if (nmax > 1) ties++;
        bq_zero |= gt_pl(p, &L, ridx, alt, pl); /* get_germ_gq(alt 1-char): that allele is skipped */
        int gq2, tie2;
        argmin_gt(pl, &gq2, &tie2);
        if (gq2 < p->min_gq) { log[10] += tri_sum; continue; }
        if (!(ref_count >= p->min_ref_count && cnt[alt] >= p->min_alt_count)) { log[9] += tri_sum; continue; }
      }
      ref_tri[tri] += 1;
      ccs_tri[tri] += tri_sum;
      log[13] += tri_sum;
      track_add(&track, (uint32_t)ci, rpos, (uint32_t)tri_sum);
    }
    free(callable); free(hapcnt);
    pile_free(&P);
  }
done:
  if (qseen) /* as in orc_call_chunks_seen */
    for (size_t q = 0; q <= (size_t)max_qid && q < qseen_cap; q++) qseen[q] = (uint8_t)bitset_get(&seen, q);
  free(F); free(hap); free(mm); free(seen.w);
  if (n_alt_tie) *n_alt_tie = ties;
  if (n_runs) *n_runs = track.n;
  if (rc != HM_OK) return rc;
  if (track.n > track.cap) return HM_ERR_CAPACITY;
  return bq_zero ? HM_ERR_BQ_ZERO : HM_OK;
}
