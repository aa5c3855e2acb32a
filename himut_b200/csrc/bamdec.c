/*
 * bamdec.c — native BAM region -> packed hm_read_batch decoder (host side, no CUDA).
 *
 * Replaces, for the GPU workers, what the reference does per record through pysam/htslib and
 * Python: alignments.fetch(chrom, start, end) (src/himut/caller.py:299) + bamlib.BAM.__init__
 * (src/himut/bamlib.py:15-32) + the regex walk of cslib.cs2lst / cs2tuple
 * (src/himut/cslib.py:7-44).  Same rules as himut_b200/bamio.py + pack.py (which stay as the
 * readable specification and are compared against this file in tests/test_host.py):
 *   - records overlapping [start, end) of the contig, file order, secondary (0x100) skipped,
 *     supplementary kept;
 *   - coordinates from the CIGAR, query span and reference span cross-checked against cs;
 *   - inputs the reference would crash on are rejected with a message (no cs tag, missing
 *     qualities, hard clips, read base outside ACGT under a cs match, '~' introns).
 * BGZF blocks are inflated by a small pthread pool; parsing is a single pass.
 */
#define _GNU_SOURCE
#include <pthread.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <time.h>
#include <zlib.h>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif

#include "../../include/himut_io.h"
#include "inflate_fast.h"
#include "crc32_clmul.h"
#include "bamerr.h"

/* crc32(0, p, n) of zlib: carry-less-multiply folding over the multiple-of-16 body when the CPU has it
 * (crc32_clmul.h), zlib for the tail and everywhere else */
static uint32_t block_crc(const uint8_t* p, size_t n) {
#if HM_CRC32_CLMUL
  if (n >= 64 && hm_crc32_available()) {
    size_t used = 0;
    const uint32_t state = hm_crc32_fold(0xffffffffu, p, n, &used);
    return (uint32_t)crc32((uLong)(uint32_t)~state, p + used, (uInt)(n - used));
  }
#endif
  return (uint32_t)crc32(crc32(0L, Z_NULL, 0), p, (uInt)n);
}
uint32_t hm_crc32_test(const uint8_t* p, size_t n) { return block_crc(p, n); }


/* one bin of a BAI or CSI: its smallest chunk begin, its largest chunk end and (CSI) its loffset */
typedef struct {
  uint32_t id;
  uint64_t beg, end, loff;
} idx_bin_t;

typedef struct {
  char* name;
  int32_t len;
  uint64_t* lin; /* BAI linear index */
  int32_t n_lin;
  int has_index;
  idx_bin_t* bins; /* ascending ids, the pseudo-bin left out */
  int32_t n_bin;
  uint64_t min_beg; /* smallest chunk begin of the contig */
} bam_ref_t;

typedef struct {
  uint64_t* keys_hash;
  uint32_t* ids;
  char** names;
  uint32_t cap, n;
} qtab_t;

typedef struct hm_bam {
  FILE* f;
  const uint8_t* map;  /* the whole file, mapped read-only (NULL: read() path) */
  size_t map_len;
  char* path;
  char* header;
  int32_t n_ref;
  bam_ref_t* refs;
  uint64_t first_record; /* virtual offset */
  uint64_t file_size;
  int index_kind;        /* HM_BAM_INDEX_NONE / _BAI / _CSI */
  int min_shift, depth;  /* binning scheme of the index: (14, 5) for a BAI */
  qtab_t qt;
  char err[512];
  /* last decoded batch (owned) */
  hm_read_batch batch;
  int32_t *tstart, *tend, *qstart, *qlen;
  uint8_t *mapq, *flags;
  uint32_t *qname_id, *n_ops;
  uint64_t *seq_off, *bq_off, *op_off;
  uint8_t *seq, *bq;
  uint32_t* ops;
  size_t cap_reads, cap_seq, cap_bq, cap_ops;
  /* compact quality stream of the last batch (HM_BAM_OPT_COMPACT_BQ): hm_bq_compact of himut_b200.h */
  uint8_t *qmask, *qexc;
  uint64_t* qexc_off;
  size_t cap_qmask, cap_qexc, cap_qexc_off;
  uint64_t n_qexc;
  int no_seq;     /* HM_BAM_OPT_NO_SEQ: batches come without the 2-bit base stream */
  int compact_bq; /* HM_BAM_OPT_COMPACT_BQ: qualities come as modal bitmap + exceptions, built while records are parsed */
  int modal;      /* the modal quality of the handle's compact streams (0: not chosen yet) */
  /* HM_BAM_OPT_BUFFER_SET: two sets of output buffers, so that one batch can be uploaded while the next is decoded */
  struct hm_bufset {
    int32_t *tstart, *tend, *qstart, *qlen;
    uint8_t *mapq, *flags;
    uint32_t *qname_id, *n_ops;
    uint64_t *seq_off, *bq_off, *op_off;
    uint8_t *seq, *bq;
    uint32_t* ops;
    size_t cap_reads, cap_seq, cap_bq, cap_ops;
    uint8_t *qmask, *qexc;
    uint64_t* qexc_off;
    size_t cap_qmask, cap_qexc, cap_qexc_off;
    uint64_t n_qexc;
  } other; /* the set that is not active */
  int cur_set;
  /* the last hm_bam_region_plan: block table, entry points, and the compressed range when the file is not mapped */
  uint64_t *p_coff, *p_uoff, *p_entry;
  uint32_t *p_csize, *p_isize, *p_crc;
  size_t cap_plan_blocks, cap_plan_entry;
  uint8_t* p_comp;
  size_t cap_p_comp;
  /* hm_bam_set_reference: the caller's sequence of contig ref_rid (NULL: none), for records with neither cs:Z nor MD:Z */
  const uint8_t* ref_seq;
  size_t ref_len;
  int ref_rid;
} hm_bam;

/* swap the active output buffers with the parked set */
static void swap_bufset(hm_bam* b) {
  struct hm_bufset t;
#define SW(f) t.f = b->f; b->f = b->other.f; b->other.f = t.f
  SW(tstart); SW(tend); SW(qstart); SW(qlen); SW(mapq); SW(flags); SW(qname_id); SW(n_ops); SW(seq_off); SW(bq_off); SW(op_off);
  SW(seq); SW(bq); SW(ops); SW(cap_reads); SW(cap_seq); SW(cap_bq); SW(cap_ops); SW(qmask); SW(qexc); SW(qexc_off);
  SW(cap_qmask); SW(cap_qexc); SW(cap_qexc_off); SW(n_qexc);
#undef SW
}

static int fail(hm_bam* b, const char* fmt, const char* a, long x) {
  snprintf(b->err, sizeof(b->err), fmt, a ? a : "", x);
  return HM_ERR_ARG;
}

/* ------------------------------------------------------------------ qname table (FNV-1a) */
static uint64_t fnv(const char* s, size_t n) {
  uint64_t h = 1469598103934665603ull;
  for (size_t i = 0; i < n; i++) { h ^= (uint8_t)s[i]; h *= 1099511628211ull; }
  return h ? h : 1;
}
static int qt_grow(qtab_t* t) {
  uint32_t ncap = t->cap ? t->cap * 2 : 1u << 16;
  uint64_t* nk = (uint64_t*)calloc(ncap, sizeof(uint64_t));
  uint32_t* ni = (uint32_t*)malloc(ncap * sizeof(uint32_t));
  if (!nk || !ni) return -1;
  for (uint32_t i = 0; i < t->cap; i++)
    if (t->keys_hash[i]) {
      uint32_t j = (uint32_t)(t->keys_hash[i] & (ncap - 1));
      while (nk[j]) j = (j + 1) & (ncap - 1);
      nk[j] = t->keys_hash[i]; ni[j] = t->ids[i];
    }
  free(t->keys_hash); free(t->ids);
  t->keys_hash = nk; t->ids = ni; t->cap = ncap;
  return 0;
}
static int64_t qt_get(qtab_t* t, const char* s, size_t n) {
  if (t->n * 2 >= t->cap && qt_grow(t)) return -1;
  uint64_t h = fnv(s, n);
  uint32_t j = (uint32_t)(h & (t->cap - 1));
  while (t->keys_hash[j]) {
    if (t->keys_hash[j] == h) {
      const char* o = t->names[t->ids[j]];
      if (strlen(o) == n && memcmp(o, s, n) == 0) return t->ids[j];
    }
    j = (j + 1) & (t->cap - 1);
  }
  if ((t->n & 0xffff) == 0) {
    char** nn = (char**)realloc(t->names, ((size_t)t->n + 0x10000) * sizeof(char*));
    if (!nn) return -1;
    t->names = nn;
  }
  char* c = (char*)malloc(n + 1);
  if (!c) return -1;
  memcpy(c, s, n); c[n] = 0;
  t->names[t->n] = c;
  t->keys_hash[j] = h; t->ids[j] = t->n;
  return t->n++;
}

/* bytes per element of a B array tag; 0: a subtype htslib does not know (it rejects the record) */
static inline size_t b_elem_size(char sub) {
  return (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : (sub == 'i' || sub == 'I' || sub == 'f') ? 4 : 0;
}
static inline uint32_t rd32(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }

/* ------------------------------------------------------------------ BGZF */
typedef struct {
  uint64_t coff;      /* file offset of the block */
  uint32_t csize;     /* whole block size */
  uint32_t usize;     /* ISIZE */
  uint64_t uoff;      /* offset of its payload in the inflated buffer */
} blk_t;

static int read_block_header(FILE* f, uint64_t coff, blk_t* b) {
  uint8_t h[18];
  if (fseeko(f, (off_t)coff, SEEK_SET)) return -1;
  size_t got = fread(h, 1, 18, f);
  if (got == 0) return 1; /* EOF */
  if (got < 18 || h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4)) return -1;
  uint16_t xlen = (uint16_t)(h[10] | (h[11] << 8));
  uint8_t extra[4096];
  if (xlen < 6 || xlen > sizeof(extra)) return -1;
  memcpy(extra, h + 12, 6);
  if (xlen > 6 && fread(extra + 6, 1, xlen - 6, f) != (size_t)(xlen - 6)) return -1;
  int bsize = -1;
  for (int p = 0; p + 4 <= xlen;) {
    int slen = extra[p + 2] | (extra[p + 3] << 8);
    if (extra[p] == 66 && extra[p + 1] == 67 && slen == 2) bsize = extra[p + 4] | (extra[p + 5] << 8);
    p += 4 + slen;
  }
  if (bsize < 0) return -1;
  b->coff = coff; b->csize = (uint32_t)bsize + 1;
  uint8_t tail[4];
  if (fseeko(f, (off_t)(coff + b->csize - 4), SEEK_SET) || fread(tail, 1, 4, f) != 4) return -1;
  b->usize = (uint32_t)tail[0] | ((uint32_t)tail[1] << 8) | ((uint32_t)tail[2] << 16) | ((uint32_t)tail[3] << 24);
  return 0;
}

/* HIMUT_B200_DECODE_TIMING=1: seconds per phase of the last region decode, to stderr */
static double g_phase[8];
static inline double now_s(void) { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec; }

typedef struct {
  const uint8_t* comp; /* compressed bytes of the span; blocks[i].coff is relative to it */
  const blk_t* blocks;
  size_t n_blocks;
  uint8_t* out;
  size_t next;
  pthread_mutex_t mu;
  int error;
  int zlib_only; /* HIMUT_B200_ZLIB_INFLATE=1: A/B against the library decoder */
  size_t grab;   /* blocks a worker takes at a time */
} inflate_job_t;

static void* inflate_worker(void* arg) {
  inflate_job_t* j = (inflate_job_t*)arg;
  z_stream zs;
  memset(&zs, 0, sizeof(zs));
  if (inflateInit2(&zs, -15) != Z_OK) { j->error = 1; return NULL; }
  for (;;) {
    pthread_mutex_lock(&j->mu);
    size_t i0 = j->next;
    j->next += j->grab; /* a few blocks per grab */
    pthread_mutex_unlock(&j->mu);
    if (i0 >= j->n_blocks) break;
    /* own decoder first (inflate_fast.h), two blocks at a time so their dependency chains overlap; zlib when it
     * declines a block or the CRC disagrees */
    const size_t i_end = i0 + j->grab < j->n_blocks ? i0 + j->grab : j->n_blocks;
    for (size_t i = i0; i < i_end; i += 2) {
      const size_t n_here = i + 1 < i_end ? 2 : 1;
      const uint8_t* payload[2] = {NULL, NULL};
      size_t payload_len[2] = {0, 0};
      uint8_t* dst[2] = {NULL, NULL};
      uint32_t want_crc[2] = {0, 0};
      int ok[2] = {0, 0};
      for (size_t k = 0; k < n_here; k++) {
        const blk_t* b = &j->blocks[i + k];
        const uint8_t* src = j->comp + b->coff;
        const uint16_t xlen = (uint16_t)(src[10] | (src[11] << 8));
        payload[k] = src + 12 + xlen;
        payload_len[k] = b->csize - 12 - xlen - 8;
        want_crc[k] = rd32(src + b->csize - 8);
        dst[k] = j->out + b->uoff;
        if (b->usize == 0) ok[k] = 1; /* the empty end-of-file block */
      }
      if (!j->zlib_only) {
        if (n_here == 2 && !ok[0] && !ok[1]) {
          int rc[2];
          hm_inflate_raw2(payload[0], payload_len[0], dst[0], j->blocks[i].usize, payload[1], payload_len[1], dst[1], j->blocks[i + 1].usize, rc);
          ok[0] = rc[0] == 0; ok[1] = rc[1] == 0;
        } else {
          for (size_t k = 0; k < n_here; k++)
            if (!ok[k]) ok[k] = hm_inflate_raw(payload[k], payload_len[k], dst[k], j->blocks[i + k].usize) == 0;
        }
        for (size_t k = 0; k < n_here; k++)
          if (ok[k] && j->blocks[i + k].usize) ok[k] = block_crc(dst[k], j->blocks[i + k].usize) == want_crc[k];
      }
      for (size_t k = 0; k < n_here && !j->error; k++) {
        if (ok[k]) continue;
        const blk_t* b = &j->blocks[i + k];
        if (b->usize == 0) continue;
        inflateReset(&zs);
        zs.next_in = (Bytef*)payload[k];
        zs.avail_in = (uInt)payload_len[k];
        zs.next_out = dst[k];
        zs.avail_out = b->usize;
        if (inflate(&zs, Z_FINISH) != Z_STREAM_END || block_crc(dst[k], b->usize) != want_crc[k]) j->error = 1;
      }
      if (j->error) break;
    }
    if (j->error) break;
  }
  inflateEnd(&zs);
  return NULL;
}

/* sequential reader over the inflated stream: compressed spans are read in one piece, their
 * BGZF headers walked in memory, and the blocks inflated by the pool */
typedef struct {
  hm_bam* b;
  uint64_t next_coff;
  uint8_t* buf;      /* inflated bytes not yet consumed */
  size_t len, pos, cap;
  size_t span;       /* compressed bytes to read next time (grows 1 MB -> 64 MB) */
  int eof, threads;
} stream_t;

static int stream_fill(stream_t* s) {
  if (s->eof) return 1;
  if (s->span == 0) s->span = 1u << 20;
  for (;;) {
    double t0 = now_s();
    uint8_t* comp;
    size_t got;
    const int mapped = s->b->map != NULL;
    if (mapped) { /* compressed bytes straight out of the page cache */
      if (s->next_coff >= s->b->map_len) { s->eof = 1; return 1; }
      comp = (uint8_t*)(s->b->map + s->next_coff);
      got = s->b->map_len - s->next_coff < s->span ? s->b->map_len - s->next_coff : s->span;
    } else {
      comp = (uint8_t*)malloc(s->span);
      if (!comp) return -1;
      if (fseeko(s->b->f, (off_t)s->next_coff, SEEK_SET)) { free(comp); return -1; }
      got = fread(comp, 1, s->span, s->b->f);
      if (got == 0) { free(comp); s->eof = 1; return 1; }
    }
    g_phase[0] += now_s() - t0; t0 = now_s();
    size_t nb = 0, cap_b = got / 200 + 16, off = 0;
    uint64_t usum = 0;
    blk_t* blocks = (blk_t*)malloc(cap_b * sizeof(blk_t));
    if (!blocks) { if (!mapped) free(comp); return -1; }
    int bad = 0;
    while (off + 18 <= got) {
      const uint8_t* h = comp + off;
      if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4)) { bad = 1; break; }
      uint16_t xlen = (uint16_t)(h[10] | (h[11] << 8));
      if (off + 12 + xlen > got) break;
      int bsize = -1;
      for (int q = 0; q + 4 <= xlen;) {
        int slen = h[12 + q + 2] | (h[12 + q + 3] << 8);
        if (h[12 + q] == 66 && h[12 + q + 1] == 67 && slen == 2) bsize = h[12 + q + 4] | (h[12 + q + 5] << 8);
        q += 4 + slen;
      }
      if (bsize < 0) { bad = 1; break; }
      size_t csize = (size_t)bsize + 1;
      if (off + csize > got) break;
      if (nb == cap_b) { cap_b *= 2; blk_t* nbk = (blk_t*)realloc(blocks, cap_b * sizeof(blk_t)); if (!nbk) { bad = 1; break; } blocks = nbk; }
      blocks[nb].coff = off; blocks[nb].csize = (uint32_t)csize; blocks[nb].usize = rd32(h + csize - 4); blocks[nb].uoff = usum;
      usum += blocks[nb].usize; off += csize; nb++;
    }
    if (bad) { free(blocks); if (!mapped) free(comp); return -1; }
    if (nb == 0) { /* a block larger than the span, or a truncated file */
      free(blocks); if (!mapped) free(comp);
      if (got < s->span) return -1;
      s->span *= 2;
      continue;
    }
    size_t keep = s->len - s->pos;
    if (s->pos && keep) memmove(s->buf, s->buf + s->pos, keep);
    s->len = keep; s->pos = 0;
    if (s->len + usum > s->cap) {
      size_t nc = s->len + usum + (1 << 20);
      uint8_t* nbuf = (uint8_t*)realloc(s->buf, nc);
      if (!nbuf) { free(blocks); if (!mapped) free(comp); return -1; }
      s->buf = nbuf; s->cap = nc;
    }
    g_phase[1] += now_s() - t0; t0 = now_s();
    inflate_job_t job;
    memset(&job, 0, sizeof(job));
    job.comp = comp; job.blocks = blocks; job.n_blocks = nb; job.out = s->buf + s->len;
    job.zlib_only = getenv("HIMUT_B200_ZLIB_INFLATE") != NULL;
    pthread_mutex_init(&job.mu, NULL);
    int nt = s->threads < 1 ? 1 : (s->threads > 64 ? 64 : s->threads);
    job.grab = nb / ((size_t)nt * 8) + 1; /* about eight grabs per thread: balanced, few lock round trips */
    if (job.grab > 16) job.grab = 16;
    if ((size_t)nt > (nb + job.grab - 1) / job.grab) nt = (int)((nb + job.grab - 1) / job.grab);
    pthread_t th[64];
    for (int t = 1; t < nt; t++) pthread_create(&th[t], NULL, inflate_worker, &job);
    inflate_worker(&job);
    for (int t = 1; t < nt; t++) pthread_join(th[t], NULL);
    pthread_mutex_destroy(&job.mu);
    g_phase[2] += now_s() - t0; t0 = now_s();
    if (!mapped) free(comp);
    free(blocks);
    g_phase[3] += now_s() - t0;
    if (job.error) return -1;
    s->len += usum;
    s->next_coff += off;
    if (s->span < (64u << 20)) s->span *= 2;
    return 0;
  }
}
/* make `n` bytes available at buf+pos; 0 ok, 1 EOF, -1 error */
static int stream_need(stream_t* s, size_t n) {
  while (s->len - s->pos < n) {
    int rc = stream_fill(s);
    if (rc) return (s->len - s->pos >= n) ? 0 : rc;
  }
  return 0;
}
static int stream_seek(stream_t* s, uint64_t voffset) {
  s->next_coff = voffset >> 16;
  s->len = s->pos = 0; s->eof = 0;
  int rc = stream_fill(s);
  if (rc < 0) return rc;
  s->pos = voffset & 0xffff;
  return 0;
}

/* ------------------------------------------------------------------ open / close */
/* the binning scheme of SAM spec 5.3, for an index of min_shift and depth (a BAI is (14, 5)): level l has 8^l bins of
 * 2^(min_shift + 3 (depth - l)) positions, numbered from bin_first(l); the pseudo-bin follows the last level */
static inline uint32_t bin_first(int level) { return (uint32_t)(((1ull << (3 * level)) - 1) / 7); }
static inline uint32_t pseudo_bin(int depth) { return bin_first(depth + 1) + 1; }
static int bin_level(uint32_t bin) {
  int l = 0;
  while (bin >= bin_first(l + 1)) l++;
  return l;
}
/* first reference position of a bin, and the number of positions it covers */
static int64_t bin_start(uint32_t bin, int min_shift, int depth) {
  const int l = bin_level(bin);
  return (int64_t)(bin - bin_first(l)) << (min_shift + 3 * (depth - l));
}
static int64_t bin_size(uint32_t bin, int min_shift, int depth) { return (int64_t)1 << (min_shift + 3 * (depth - bin_level(bin))); }

static char* path_with(const char* base, size_t n, const char* ext) {
  char* p = (char*)malloc(n + strlen(ext) + 1);
  if (p) { memcpy(p, base, n); strcpy(p + n, ext); }
  return p;
}

/* the payload of a BGZF-compressed file (a CSI), NULL with b->err set when it is not one */
static uint8_t* bgzf_slurp(hm_bam* b, const uint8_t* d, size_t sz, const char* ip, size_t* out_len) {
  size_t cap = 1u << 16, n = 0, off = 0;
  uint8_t* u = (uint8_t*)malloc(cap);
  z_stream zs;
  memset(&zs, 0, sizeof(zs));
  if (!u || inflateInit2(&zs, -15) != Z_OK) { free(u); snprintf(b->err, sizeof(b->err), "out of memory reading %s", ip); return NULL; }
  while (off < sz) {
    const uint8_t* h = d + off;
    int bsize = -1;
    if (sz - off >= 18 && h[0] == 0x1f && h[1] == 0x8b && h[2] == 8 && (h[3] & 4)) {
      const size_t xlen = (size_t)(h[10] | (h[11] << 8));
      for (size_t q = 0; 12 + xlen <= sz - off && q + 4 <= xlen;) {
        const size_t slen = (size_t)(h[12 + q + 2] | (h[12 + q + 3] << 8));
        if (h[12 + q] == 66 && h[12 + q + 1] == 67 && slen == 2 && q + 6 <= xlen) bsize = h[12 + q + 4] | (h[12 + q + 5] << 8);
        q += 4 + slen;
      }
      if (bsize >= 0 && ((size_t)bsize + 1 < 12 + xlen + 8 || (size_t)bsize + 1 > sz - off)) bsize = -1;
      if (bsize >= 0) {
        const size_t csize = (size_t)bsize + 1, isize = rd32(h + csize - 4);
        if (isize > 65536) goto bad;
        if (n + isize > cap) {
          while (n + isize > cap) cap *= 2;
          uint8_t* nu = (uint8_t*)realloc(u, cap);
          if (!nu) goto bad;
          u = nu;
        }
        inflateReset(&zs);
        zs.next_in = (Bytef*)(h + 12 + xlen); zs.avail_in = (uInt)(csize - 12 - xlen - 8);
        zs.next_out = u + n; zs.avail_out = (uInt)isize;
        if ((isize || csize - 12 - xlen - 8 > 2) && (inflate(&zs, Z_FINISH) != Z_STREAM_END || zs.avail_out || block_crc(u + n, isize) != rd32(h + csize - 8))) bsize = -1;
        else { n += isize; off += csize; continue; }
      }
    }
  bad:
    inflateEnd(&zs);
    free(u);
    snprintf(b->err, sizeof(b->err), "%s is not a BGZF-compressed CSI index (block at byte %zu)", ip, off);
    return NULL;
  }
  inflateEnd(&zs);
  *out_len = n;
  return u;
}

static int cmp_u64(const void* x, const void* y) {
  const uint64_t a = *(const uint64_t*)x, c = *(const uint64_t*)y;
  return a < c ? -1 : a > c;
}
static int cmp_bin(const void* x, const void* y) {
  const uint32_t a = ((const idx_bin_t*)x)->id, c = ((const idx_bin_t*)y)->id;
  return a < c ? -1 : a > c;
}

/* the bins of one reference at d + *q (n_bin, then per bin: bin, [loffset,] n_chunk, chunks), every count bounded by
 * the bytes left; R NULL: parsed and checked, not kept (references past the BAM's) */
static int load_bins(hm_bam* b, bam_ref_t* R, const uint8_t* d, size_t sz, size_t* qp, int csi, const char* ip) {
  const uint32_t pseudo = pseudo_bin(b->depth);
  const size_t fixed = csi ? 16 : 8; /* bin, loffset (CSI), n_chunk */
  size_t q = *qp;
#define IDX_BAD(...) do { int k_ = snprintf(b->err, sizeof(b->err), "%s: ", ip); snprintf(b->err + k_, sizeof(b->err) - (size_t)k_, __VA_ARGS__); return -1; } while (0)
  if (sz - q < 4) IDX_BAD("truncated at byte %zu (n_bin)", q);
  const int32_t nbin = (int32_t)rd32(d + q);
  q += 4;
  if (nbin < 0 || (size_t)nbin > (sz - q) / fixed) IDX_BAD("n_bin %d runs past the end of the index", nbin);
  if (R) {
    R->bins = (idx_bin_t*)malloc(((size_t)nbin + 1) * sizeof(idx_bin_t));
    if (!R->bins) IDX_BAD("out of memory for %d bins", nbin);
    R->min_beg = UINT64_MAX;
  }
  for (int32_t k = 0; k < nbin; k++) {
    if (sz - q < fixed) IDX_BAD("truncated at byte %zu (bin)", q);
    const uint32_t bin = rd32(d + q);
    uint64_t loff = 0;
    if (csi) memcpy(&loff, d + q + 4, 8);
    const int32_t nchunk = (int32_t)rd32(d + q + fixed - 4);
    q += fixed;
    if (csi && (bin > pseudo || bin == pseudo - 1)) IDX_BAD("bin %u past the pseudo-bin %u", bin, pseudo); /* pseudo - 1: past the last level */
    if (csi && bin != pseudo && (loff >> 16) >= b->file_size) IDX_BAD("loffset of bin %u points past the end of the BAM", bin);
    if (nchunk < 0 || (size_t)nchunk > (sz - q) / 16) IDX_BAD("n_chunk %d of bin %u runs past the end of the index", nchunk, bin);
    uint64_t e = 0, bg = UINT64_MAX;
    for (int32_t c = 0; c < nchunk; c++) {
      uint64_t cb, ce;
      memcpy(&cb, d + q + 16 * (size_t)c, 8); memcpy(&ce, d + q + 16 * (size_t)c + 8, 8);
      if (csi && bin != pseudo && cb > ce) IDX_BAD("chunk %d of bin %u begins after its end", c, bin);
      if (csi && bin != pseudo && (cb >> 16) >= b->file_size) IDX_BAD("chunk %d of bin %u points past the end of the BAM", c, bin);
      if (ce > e) e = ce;
      if (cb < bg) bg = cb;
    }
    q += 16 * (size_t)nchunk;
    if (R && bin < pseudo - 1 && nchunk) {
      idx_bin_t* x = &R->bins[R->n_bin++];
      x->id = bin; x->beg = bg; x->end = e; x->loff = loff;
      if (bg < R->min_beg) R->min_beg = bg;
    }
  }
#undef IDX_BAD
  if (R) qsort(R->bins, (size_t)R->n_bin, sizeof(idx_bin_t), cmp_bin);
  *qp = q;
  return 0;
}

/* the index of the BAM, by the names htslib finds: <bam>.bai, <bam>.csi, then <stem>.bai and <stem>.csi for x.bam.
 * None found: b->index_kind stays 0 and every query scans from the first record.  -1 (b->err set): an index that
 * cannot be read. */
static int load_index(hm_bam* b) {
  const size_t n = strlen(b->path);
  const size_t stem = n > 4 && strcmp(b->path + n - 4, ".bam") == 0 ? n - 4 : 0;
  const struct { size_t len; const char* ext; int kind; } cand[4] = {
      {n, ".bai", HM_BAM_INDEX_BAI}, {n, ".csi", HM_BAM_INDEX_CSI}, {stem, ".bai", HM_BAM_INDEX_BAI}, {stem, ".csi", HM_BAM_INDEX_CSI}};
  FILE* f = NULL;
  char* ip = NULL;
  int kind = 0;
  for (int i = 0; i < 4 && !f; i++) {
    if (!cand[i].len) continue;
    free(ip);
    ip = path_with(b->path, cand[i].len, cand[i].ext);
    if (!ip) return -1;
    f = fopen(ip, "rb");
    kind = cand[i].kind;
  }
  if (!f) { free(ip); return 0; }
  size_t sz = 0;
  uint8_t* raw = NULL;
  if (fseeko(f, 0, SEEK_END) == 0) {
    const off_t end = ftello(f);
    sz = end > 0 ? (size_t)end : 0;
    raw = (uint8_t*)malloc(sz + 8);
    if (raw && (fseeko(f, 0, SEEK_SET) || fread(raw, 1, sz, f) != sz)) { free(raw); raw = NULL; }
  }
  fclose(f);
  int rc = -1;
  uint8_t* d = raw;
  if (!raw) { snprintf(b->err, sizeof(b->err), "cannot read %s", ip); goto out; }
  b->min_shift = 14; b->depth = 5;
  size_t q;
  int32_t nref;
  if (kind == HM_BAM_INDEX_BAI) {
    if (sz < 8 || memcmp(d, "BAI\1", 4)) { snprintf(b->err, sizeof(b->err), "%s is not a BAI index", ip); goto out; }
    nref = (int32_t)rd32(d + 4);
    q = 8;
  } else {
    d = bgzf_slurp(b, raw, sz, ip, &sz);
    if (!d) goto out;
    if (sz < 16 || memcmp(d, "CSI\1", 4)) { snprintf(b->err, sizeof(b->err), "%s is not a CSI index", ip); goto out; }
    const int32_t ms = (int32_t)rd32(d + 4), depth = (int32_t)rd32(d + 8), l_aux = (int32_t)rd32(d + 12);
    if (ms < 1 || depth < 0 || depth > 10 || ms + 3 * depth > 62) {
      snprintf(b->err, sizeof(b->err), "%s: unsupported min_shift %d / depth %d", ip, ms, depth);
      goto out;
    }
    b->min_shift = ms; b->depth = depth;
    for (int32_t r = 0; r < b->n_ref; r++)
      if ((int64_t)b->refs[r].len > ((int64_t)1 << (ms + 3 * depth))) {
        snprintf(b->err, sizeof(b->err), "%s: min_shift %d and depth %d cover %lld positions, %s has %d", ip, ms, depth,
                 (long long)1 << (ms + 3 * depth), b->refs[r].name, b->refs[r].len);
        goto out;
      }
    if (l_aux < 0 || (size_t)l_aux > sz - 16 || sz - 16 - (size_t)l_aux < 4) { snprintf(b->err, sizeof(b->err), "%s: l_aux %d runs past the end of the index", ip, l_aux); goto out; }
    q = 16 + (size_t)l_aux;
    nref = (int32_t)rd32(d + q);
    q += 4;
  }
  if (nref < 0) { snprintf(b->err, sizeof(b->err), "%s: n_ref %d", ip, nref); goto out; }
  for (int32_t r = 0; r < nref; r++) {
    bam_ref_t* R = r < b->n_ref ? &b->refs[r] : NULL;
    if (kind == HM_BAM_INDEX_BAI && !R) break; /* as before: references past the BAM's are not read */
    if (load_bins(b, R, d, sz, &q, kind == HM_BAM_INDEX_CSI, ip)) goto out;
    if (kind == HM_BAM_INDEX_CSI) { if (R) R->has_index = R->n_bin > 0; continue; }
    if (sz - q < 4) { snprintf(b->err, sizeof(b->err), "%s: truncated at byte %zu (n_intv)", ip, q); goto out; }
    const int32_t nintv = (int32_t)rd32(d + q);
    q += 4;
    if (nintv < 0 || (size_t)nintv > (sz - q) / 8) { snprintf(b->err, sizeof(b->err), "%s: n_intv %d runs past the end of the index", ip, nintv); goto out; }
    R->lin = (uint64_t*)malloc(((size_t)nintv + 1) * 8);
    if (!R->lin) { snprintf(b->err, sizeof(b->err), "out of memory reading %s", ip); goto out; }
    R->n_lin = nintv;
    R->has_index = (R->n_bin || nintv);
    memcpy(R->lin, d + q, 8 * (size_t)nintv);
    q += 8 * (size_t)nintv;
  }
  b->index_kind = kind;
  rc = 0;
out:
  if (d != raw) free(d);
  free(raw);
  free(ip);
  return rc;
}

/* the virtual offset the records of [start, ...) of contig rid are read from; 0: the index knows no record of the
 * contig.  BAI: the linear-index entry of start's 16 kb window, or of the nearest window to its left that has one.
 * CSI (htslib's hts_itr_query): the loffset of the leaf bin that holds start, else of its nearest left sibling, else
 * of its parent, and so on up; without one, the contig's first chunk.  Without an index: the first record. */
static uint64_t seek_voff(const hm_bam* b, int rid, int32_t start) {
  if (!b->index_kind) return b->first_record;
  const bam_ref_t* R = &b->refs[rid];
  if (!R->has_index) return 0;
  if (b->index_kind == HM_BAM_INDEX_BAI) {
    int32_t w = start >> 14;
    if (w >= R->n_lin) w = R->n_lin - 1;
    uint64_t v = 0;
    for (; w >= 0 && !v; w--) v = R->lin[w];
    return v ? v : b->first_record;
  }
  const int64_t top = ((int64_t)1 << (b->min_shift + 3 * b->depth)) - 1;
  uint32_t bin = bin_first(b->depth) + (uint32_t)(((int64_t)start < top ? (int64_t)start : top) >> b->min_shift);
  for (;;) {
    size_t lo = 0, hi = (size_t)R->n_bin;
    while (lo < hi) { const size_t m = (lo + hi) / 2; if (R->bins[m].id < bin) lo = m + 1; else hi = m; }
    if (lo < (size_t)R->n_bin && R->bins[lo].id == bin && R->bins[lo].loff) return R->bins[lo].loff;
    if (bin == 0) break;
    const uint32_t first = (((bin - 1) >> 3) << 3) + 1; /* the first child of the parent */
    bin = bin > first ? bin - 1 : (bin - 1) >> 3;
  }
  return R->min_beg;
}

void hm_bam_close(hm_bam* b) {
  if (!b) return;
  if (b->map) munmap((void*)b->map, b->map_len);
  if (b->f) fclose(b->f);
  for (int32_t i = 0; i < b->n_ref; i++) { free(b->refs[i].name); free(b->refs[i].lin); free(b->refs[i].bins); }
  free(b->refs); free(b->header); free(b->path);
  free(b->p_coff); free(b->p_uoff); free(b->p_entry); free(b->p_csize); free(b->p_isize); free(b->p_crc); free(b->p_comp);
  for (uint32_t i = 0; i < b->qt.n; i++) free(b->qt.names[i]);
  free(b->qt.names); free(b->qt.keys_hash); free(b->qt.ids);
  for (int k = 0; k < 2; k++) { /* both buffer sets */
    free(b->tstart); free(b->tend); free(b->qstart); free(b->qlen); free(b->mapq); free(b->flags); free(b->qname_id);
    free(b->n_ops); free(b->seq_off); free(b->bq_off); free(b->op_off); free(b->seq); free(b->bq); free(b->ops);
    free(b->qmask); free(b->qexc); free(b->qexc_off);
    swap_bufset(b);
  }
  free(b);
}

#if defined(__x86_64__) && defined(__GNUC__)
static int have_ssse3(void); /* probed once in hm_bam_open, read by the record-decode threads */
#endif

/* why the last hm_bam_open of this thread failed: hm_bam_error(NULL) */
static __thread char g_open_err[512];

int hm_bam_open(const char* path, hm_bam** out) {
  if (!path || !out) return HM_ERR_ARG;
  *out = NULL;
  g_open_err[0] = 0;
  (void)hi_use_run(); (void)hm_crc32_available(); /* one-time CPU probes and tables, before any worker thread exists */
#if defined(__x86_64__) && defined(__GNUC__)
  (void)have_ssse3();
#endif
  hm_bam* b = (hm_bam*)calloc(1, sizeof(hm_bam));
  if (!b) return HM_ERR_ARG;
  b->path = strdup(path);
  b->f = fopen(path, "rb");
  if (!b->f) { hm_bam_close(b); return HM_ERR_ARG; }
  {
    struct stat st;
    if (fstat(fileno(b->f), &st) == 0) b->file_size = (uint64_t)st.st_size;
    if (b->file_size > 0) {
      void* m = mmap(NULL, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fileno(b->f), 0);
      if (m != MAP_FAILED) { b->map = (const uint8_t*)m; b->map_len = (size_t)st.st_size; }
    }
  }
  stream_t s;
  memset(&s, 0, sizeof(s));
  s.b = b; s.threads = 1;
  int rc = HM_ERR_ARG;
  if (stream_seek(&s, 0) || stream_need(&s, 12) || memcmp(s.buf + s.pos, "BAM\1", 4)) goto done;
  {
    uint32_t ltext = rd32(s.buf + s.pos + 4);
    if (stream_need(&s, 12 + (size_t)ltext)) goto done;
    b->header = (char*)malloc((size_t)ltext + 1);
    memcpy(b->header, s.buf + s.pos + 8, ltext); b->header[ltext] = 0;
    b->n_ref = (int32_t)rd32(s.buf + s.pos + 8 + ltext);
    size_t consumed = 12 + (size_t)ltext;
    b->refs = (bam_ref_t*)calloc((size_t)b->n_ref + 1, sizeof(bam_ref_t));
    for (int32_t i = 0; i < b->n_ref; i++) {
      if (stream_need(&s, consumed + 4)) goto done;
      uint32_t ln = rd32(s.buf + s.pos + consumed);
      if (stream_need(&s, consumed + 8 + ln)) goto done;
      b->refs[i].name = (char*)malloc(ln + 1);
      memcpy(b->refs[i].name, s.buf + s.pos + consumed + 4, ln); b->refs[i].name[ln] = 0;
      b->refs[i].len = (int32_t)rd32(s.buf + s.pos + consumed + 4 + ln);
      consumed += 8 + ln;
    }
    /* virtual offset of the first record: walk the blocks again, cheaply */
    uint64_t coff = 0, left = consumed;
    for (;;) {
      blk_t blk;
      if (read_block_header(b->f, coff, &blk)) goto done;
      if (left < blk.usize) { b->first_record = (coff << 16) | left; break; }
      if (left == blk.usize) { b->first_record = ((coff + blk.csize) << 16); break; }
      left -= blk.usize; coff += blk.csize;
    }
  }
  if (load_index(b) < 0) goto done;
  rc = HM_OK;
done:
  free(s.buf);
  if (rc) {
    snprintf(g_open_err, sizeof(g_open_err), "%s", b->err);
    hm_bam_close(b);
    return rc;
  }
  *out = b;
  return HM_OK;
}

const char* hm_bam_error(const hm_bam* b) { return b ? b->err : g_open_err; }
int hm_bam_index_kind(const hm_bam* b) { return b ? b->index_kind : HM_BAM_INDEX_NONE; }
const char* hm_bam_header_text(const hm_bam* b) { return b->header; }
int hm_bam_n_refs(const hm_bam* b) { return b->n_ref; }
const char* hm_bam_ref_name(const hm_bam* b, int i) { return (i >= 0 && i < b->n_ref) ? b->refs[i].name : NULL; }
int hm_bam_ref_len(const hm_bam* b, int i) { return (i >= 0 && i < b->n_ref) ? b->refs[i].len : -1; }
int hm_bam_set_reference(hm_bam* b, int rid, const uint8_t* seq, size_t len) {
  if (!b) return HM_ERR_ARG;
  b->ref_seq = NULL; b->ref_len = 0; b->ref_rid = -1;
  if (!seq) return HM_OK;
  if (rid < 0 || rid >= b->n_ref) return fail(b, "invalid contig index%s %ld", NULL, rid);
  if ((uint64_t)len != (uint64_t)b->refs[rid].len) {
    snprintf(b->err, sizeof(b->err), "the reference sequence of %s has %zu bases, its @SQ LN %d", b->refs[rid].name, len, b->refs[rid].len);
    return HM_ERR_ARG;
  }
  b->ref_seq = seq; b->ref_len = len; b->ref_rid = rid;
  return HM_OK;
}
uint32_t hm_bam_n_qnames(const hm_bam* b) { return b->qt.n; }
const char* hm_bam_qname(const hm_bam* b, uint32_t id) { return id < b->qt.n ? b->qt.names[id] : NULL; }
/* the names whose flag is set, each followed by '\n', in id order: what a worker that owns only a run of a contig's
 * chunks hands to the merge, which counts distinct names per contig (m.num_ccs, caller.py:318-320) across runs */
int hm_bam_qnames_blob(const hm_bam* b, const uint8_t* flags, size_t n_flags, char* out, size_t cap, size_t* need) {
  if (!b || !need || (n_flags && !flags)) return HM_ERR_ARG;
  size_t n = 0;
  const size_t lim = n_flags < b->qt.n ? n_flags : b->qt.n;
  for (size_t i = 0; i < lim; i++) {
    if (!flags[i]) continue;
    const size_t l = strlen(b->qt.names[i]);
    if (out && n + l + 1 <= cap) { memcpy(out + n, b->qt.names[i], l); out[n + l] = '\n'; }
    n += l + 1;
  }
  *need = n;
  return (out && n <= cap) ? HM_OK : HM_ERR_CAPACITY;
}

/* ------------------------------------------------------------------ decode */
#define GROW(ptr, cap, need, type)                                    \
  do {                                                                \
    if ((need) > (cap)) {                                             \
      size_t nc_ = (cap) ? (cap) : 1024;                              \
      while (nc_ < (need)) nc_ += nc_ / 2 + 1024;                     \
      type* np_ = (type*)realloc((ptr), nc_ * sizeof(type));          \
      if (!np_) return fail(b, "out of memory%s (%ld)", NULL, (long)nc_); \
      (ptr) = np_; (cap) = nc_;                                       \
    }                                                                 \
  } while (0)

static const int8_t NIB2CODE[16] = {-1, 0, 3, -1, 2, -1, -1, -1, 1, -1, -1, -1, -1, -1, -1, -1}; /* A1 C2 G4 T8 -> A0 T1 G2 C3 */
static inline int base_code(char c) {
  switch (c) { case 'A': case 'a': return 0; case 'T': case 't': return 1; case 'G': case 'g': return 2; case 'C': case 'c': return 3; default: return -1; }
}

/* one selected record between the serial scan (phase A) and the parallel decode (phase B) */
typedef struct {
  const uint8_t* rec;   /* start of the fixed part (after block_size) */
  const char* cs;       /* the cs:Z value, or NULL: the ops come from CIGAR + md */
  const char* md;       /* the MD:Z value, or NULL with cs NULL too: the ops come from CIGAR + the reference (ref_walk) */
  uint32_t* ext;        /* CIGAR + reference: the ops, allocated by the decode (no slot is reserved for them) */
  int32_t pos, l_seq, lead, trail, ref_span;
  size_t seq_off, bq_off, op_slot; /* where its outputs go; op_slot is an upper-bound slot, compacted afterwards */
  size_t exc_slot;                 /* compact qualities: upper-bound slot of the exceptions, compacted afterwards */
  uint32_t n_ops, n_exc;
  int32_t rspan;
  int err;              /* 0 ok, else index into the message table below */
  long err_arg;
} rec_t;


typedef struct {
  hm_bam* b;
  rec_t* recs;
  size_t n, next;
  pthread_mutex_t mu;
} decode_job_t;

/* BAM's 4-bit bases -> one code per byte (A0 T1 G2 C3, 0xff anything else); 32 bases per step with a byte shuffle */
static void nib_to_codes_scalar(const uint8_t* seq4, int32_t i, int32_t l_seq, uint8_t* codes) {
  if (i & 1) { codes[i] = (uint8_t)NIB2CODE[seq4[i >> 1] & 15]; i++; }
  for (; i + 1 < l_seq; i += 2) { const uint8_t by = seq4[i >> 1]; codes[i] = (uint8_t)NIB2CODE[by >> 4]; codes[i + 1] = (uint8_t)NIB2CODE[by & 15]; }
  if (i < l_seq) codes[i] = (uint8_t)NIB2CODE[seq4[i >> 1] >> 4];
}
/* codes -> 2-bit packed (base i at bits 2*(i&3) of byte i>>2); codes outside 0..3 (soft clips only: the caller has
 * rejected them under a match) are stored as 0, like the Python packer */
static void pack_codes_scalar(const uint8_t* codes, int32_t i, int32_t l_seq, uint8_t* dst) {
  for (; i + 3 < l_seq; i += 4) {
    uint8_t v = 0;
    for (int k = 0; k < 4; k++) { const uint8_t c = codes[i + k]; v |= (uint8_t)((c > 3 ? 0 : c) << (2 * k)); }
    dst[i >> 2] = v;
  }
  if (i < l_seq) { uint8_t v = 0; for (int32_t k = i; k < l_seq; k++) { const uint8_t c = codes[k]; v |= (uint8_t)((c > 3 ? 0 : c) << (2 * (k & 3))); } dst[i >> 2] = v; }
}
#if defined(__x86_64__) && defined(__GNUC__)
#include <immintrin.h>
static int have_ssse3(void) { static int k = -1; if (k < 0) k = __builtin_cpu_supports("ssse3") && __builtin_cpu_supports("sse4.1"); return k; }
__attribute__((target("ssse3,sse4.1"))) static int32_t nib_to_codes_simd(const uint8_t* seq4, int32_t l_seq, uint8_t* codes) {
  const __m128i lut = _mm_setr_epi8(-1, 0, 3, -1, 2, -1, -1, -1, 1, -1, -1, -1, -1, -1, -1, -1);
  const __m128i low = _mm_set1_epi8(0x0f);
  int32_t i = 0;
  for (; i + 32 <= l_seq; i += 32) {
    const __m128i v = _mm_loadu_si128((const __m128i*)(seq4 + (i >> 1)));
    const __m128i first = _mm_shuffle_epi8(lut, _mm_and_si128(_mm_srli_epi16(v, 4), low)); /* high nibble = even base */
    const __m128i second = _mm_shuffle_epi8(lut, _mm_and_si128(v, low));
    _mm_storeu_si128((__m128i*)(codes + i), _mm_unpacklo_epi8(first, second));
    _mm_storeu_si128((__m128i*)(codes + i + 16), _mm_unpackhi_epi8(first, second));
  }
  return i;
}
__attribute__((target("ssse3,sse4.1"))) static int32_t pack_codes_simd(const uint8_t* codes, int32_t l_seq, uint8_t* dst) {
  const __m128i w8 = _mm_set1_epi16(0x0401);      /* c0 + 4 c1 per byte pair  */
  const __m128i w16 = _mm_set1_epi32(0x00100001); /* p0 + 16 p1 per word pair */
  const __m128i three = _mm_set1_epi8(3);
  int32_t i = 0;
  for (; i + 16 <= l_seq; i += 16) {
    __m128i c = _mm_loadu_si128((const __m128i*)(codes + i));
    c = _mm_and_si128(_mm_andnot_si128(_mm_cmplt_epi8(c, _mm_setzero_si128()), c), three); /* 0xff (negative) -> 0 */
    const __m128i p = _mm_maddubs_epi16(c, w8);  /* 8 x (c0 | c1 << 2)            */
    const __m128i q = _mm_madd_epi16(p, w16);    /* 4 x (p0 | p1 << 4) = one byte */
    const __m128i b = _mm_packus_epi16(_mm_packus_epi32(q, q), _mm_setzero_si128());
    const uint32_t out = (uint32_t)_mm_cvtsi128_si32(b);
    memcpy(dst + (i >> 2), &out, 4);
  }
  return i;
}
#else
static int have_ssse3(void) { return 0; }
static int32_t nib_to_codes_simd(const uint8_t* seq4, int32_t l_seq, uint8_t* codes) { (void)seq4; (void)l_seq; (void)codes; return 0; }
static int32_t pack_codes_simd(const uint8_t* codes, int32_t l_seq, uint8_t* dst) { (void)codes; (void)l_seq; (void)dst; return 0; }
#endif

static inline int is_digit(char c) { return c >= '0' && c <= '9'; }
static inline int is_alpha(char c) { return (c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z'); }
/* an MD number; saturates far above any reference span, so that a huge one is left over like an exact one */
static long long md_num(const char** c) {
  long long n = 0;
  while (is_digit(**c)) { n = n * 10 + (**c - '0'); if (n > (1ll << 40)) n = 1ll << 40; (*c)++; }
  return n;
}

/* the CIGAR checks of md_walk and ref_walk (pack._check_cigar): N, P, codes past X and clips between aligned ops are
 * unsupported, the CIGAR's query length must be l_seq; 0 with R->err set on failure */
static int cigar_check(rec_t* R, const uint8_t* cig, uint32_t n_cig, int32_t l_seq) {
  uint32_t first = n_cig, last = 0; /* the aligned ops: clips may only lie outside [first, last] */
  for (uint32_t k = 0; k < n_cig; k++) { const uint32_t op = rd32(cig + 4 * k) & 15; if (op != 4 && op != 5) { if (first == n_cig) first = k; last = k; } }
  int64_t qcore = 0, qclip = 0;
  for (uint32_t k = 0; k < n_cig; k++) {
    const uint32_t c = rd32(cig + 4 * k), op = c & 15, ln = c >> 4;
    if (op == 4 || op == 5) { if (first < n_cig && k > first && k < last) { R->err = E_CIGAR_OP; R->err_arg = (long)k; return 0; } if (op == 4) qclip += ln; }
    else if (op == 0 || op == 1 || op == 7 || op == 8) qcore += ln;
    else if (op != 2) { R->err = E_CIGAR_OP; R->err_arg = (long)k; return 0; }
  }
  if (qcore + qclip != l_seq) { R->err = E_SPAN_QRY; R->err_arg = (long)qcore; return 0; }
  return 1;
}

/* a reference byte -> A0 T1 G2 C3 (either case), 0xfe anything else: never equal to a read code (0..3, 0xff) */
static inline uint8_t ref_code(uint8_t c) {
  switch (c & 0xdf) { case 'A': return 0; case 'T': return 1; case 'G': return 2; case 'C': return 3; default: return 0xfe; }
}
/* w <= 16 bases from reference bytes rp and read codes cp: bit i of *m set when read base i equals an A/C/G/T
 * reference base, of *bad when read base i is outside A/C/G/T.  16 at a time with SSE2 (only whole windows: the
 * reference may end right after the alignment), the plain loop for the rest. */
static inline void ref_masks(const uint8_t* rp, const uint8_t* cp, int w, uint32_t* m, uint32_t* bad) {
#if defined(__SSE2__)
  if (w == 16) {
    const __m128i u = _mm_and_si128(_mm_loadu_si128((const __m128i*)rp), _mm_set1_epi8((char)0xdf));
    const __m128i c = _mm_loadu_si128((const __m128i*)cp);
    const __m128i a = _mm_cmpeq_epi8(u, _mm_set1_epi8('A')), t = _mm_cmpeq_epi8(u, _mm_set1_epi8('T'));
    const __m128i g = _mm_cmpeq_epi8(u, _mm_set1_epi8('G')), cc = _mm_cmpeq_epi8(u, _mm_set1_epi8('C'));
    const __m128i acgt = _mm_or_si128(_mm_or_si128(a, t), _mm_or_si128(g, cc));
    const __m128i code = _mm_or_si128(_mm_or_si128(_mm_and_si128(t, _mm_set1_epi8(1)), _mm_and_si128(g, _mm_set1_epi8(2))),
                                      _mm_or_si128(_mm_and_si128(cc, _mm_set1_epi8(3)), _mm_andnot_si128(acgt, _mm_set1_epi8((char)0xfe))));
    *m = (uint32_t)_mm_movemask_epi8(_mm_cmpeq_epi8(code, c));
    *bad = (uint32_t)_mm_movemask_epi8(_mm_cmpeq_epi8(c, _mm_set1_epi8((char)0xff)));
    return;
  }
#endif
  uint32_t mm = 0, bb = 0;
  for (int i = 0; i < w; i++) { mm |= (uint32_t)(ref_code(rp[i]) == cp[i]) << i; bb |= (uint32_t)(cp[i] == 0xff) << i; }
  *m = mm; *bad = bb;
}

/* CIGAR + the reference sequence set with hm_bam_set_reference -> ops, the rules and the order of checks of
 * pack.parse_ref; ops needs room for 2 l_seq + n_cig + 1; 0 with R->err set on failure */
static int ref_walk(const hm_bam* b, rec_t* R, const uint8_t* cig, uint32_t n_cig, const uint8_t* codes, int32_t l_seq,
                    uint32_t* ops, uint32_t* n_out, int32_t* q_out, int32_t* rspan_out) {
#define REF_FAIL(e, a) do { R->err = (e); R->err_arg = (long)(a); return 0; } while (0)
  if (!cigar_check(R, cig, n_cig, l_seq)) return 0;
  int64_t span = 0;
  for (uint32_t k = 0; k < n_cig; k++) { const uint32_t c = rd32(cig + 4 * k), op = c & 15; if (op == 0 || op == 2 || op == 7 || op == 8) span += c >> 4; }
  if (R->pos < 0 || (uint64_t)R->pos + (uint64_t)span > (uint64_t)b->ref_len) REF_FAIL(E_REF_END, (int64_t)R->pos + span);
  const uint8_t* ref = b->ref_seq + R->pos;
  int32_t q = R->lead, r = 0;
  uint32_t n = 0, run = 0;
#define REF_FLUSH() do { if (run) { ops[n++] = HM_MAKE_OP(HM_OP_MATCH, run); run = 0; } } while (0)
  for (uint32_t k = 0; k < n_cig; k++) {
    const uint32_t cg = rd32(cig + 4 * k), op = cg & 15, ln = cg >> 4;
    if (ln == 0 || op == 4 || op == 5) continue;
    if (op == 0 || op == 7 || op == 8) {
      for (uint32_t k0 = 0; k0 < ln; k0 += 16) {
        const int w = ln - k0 < 16 ? (int)(ln - k0) : 16;
        const uint32_t full = (1u << w) - 1;
        uint32_t m, bad, sub;
        ref_masks(ref + r, codes + q, w, &m, &bad);
        if (op == 0) { /* M: mismatches are SUBs, of read bases inside A/C/G/T only */
          if (bad) REF_FAIL(E_SUB_N, q + __builtin_ctz(bad));
          sub = ~m & full;
        } else { /* =: every base matches; X: none does */
          const uint32_t stop = op == 7 ? (~m & full) : (m | bad);
          if (stop) {
            const int j = __builtin_ctz(stop);
            if ((bad >> j) & 1) REF_FAIL(op == 7 ? E_N_MATCH : E_SUB_N, q + j);
            REF_FAIL(E_REF_SPAN, r + j);
          }
          sub = op == 7 ? 0 : full;
        }
        int last = -1;
        while (sub) {
          const int j = __builtin_ctz(sub);
          sub &= sub - 1;
          run += (uint32_t)(j - last - 1);
          REF_FLUSH();
          const uint8_t rc_ = ref_code(ref[r + j]);
          ops[n++] = HM_MAKE_SUB(rc_ > 3 ? HM_BASE_N : (uint32_t)rc_, (uint32_t)codes[q + j]);
          last = j;
        }
        run += (uint32_t)(w - last - 1);
        q += w; r += w;
      }
    } else if (op == 1) {
      REF_FLUSH();
      ops[n++] = HM_MAKE_OP(HM_OP_INS, ln);
      q += (int32_t)ln;
    } else { /* D: the deleted bases are not read */
      REF_FLUSH();
      ops[n++] = HM_MAKE_OP(HM_OP_DEL, ln);
      r += (int32_t)ln;
    }
  }
  REF_FLUSH();
#undef REF_FLUSH
#undef REF_FAIL
  *n_out = n; *q_out = q; *rspan_out = r;
  return 1;
}

/* CIGAR + MD:Z -> ops, the rules and the order of checks of pack.parse_md; 0 with R->err set on failure */
static int md_walk(rec_t* R, const uint8_t* cig, uint32_t n_cig, const uint8_t* codes, int32_t l_seq, uint32_t* ops,
                   uint32_t* n_out, int32_t* q_out, int32_t* rspan_out) {
#define MD_FAIL(e, a) do { R->err = (e); R->err_arg = (long)(a); return 0; } while (0)
  if (!cigar_check(R, cig, n_cig, l_seq)) return 0;
  const char* md = R->md;
  const char* c = md;
  const char* good = md; /* end of the longest prefix the grammar accepts */
  if (is_digit(*c)) {
    while (is_digit(*c)) c++;
    good = c;
    while (*c) {
      if (*c == '^') { const char* s0 = ++c; while (is_alpha(*c)) c++; if (c == s0) break; }
      else if (is_alpha(*c)) c++;
      else break;
      if (!is_digit(*c)) break;
      while (is_digit(*c)) c++;
      good = c;
    }
  }
  if (*good || good == md) MD_FAIL(E_MD_TOKEN, good - md);
  c = md;
  long long mnum = md_num(&c);
  int32_t q = R->lead, r = 0;
  uint32_t n = 0, run = 0;
#define MD_FLUSH() do { if (run) { ops[n++] = HM_MAKE_OP(HM_OP_MATCH, run); run = 0; } } while (0)
  for (uint32_t k = 0; k < n_cig; k++) {
    const uint32_t cg = rd32(cig + 4 * k), op = cg & 15, ln = cg >> 4;
    if (ln == 0 || op == 4 || op == 5) continue;
    if (op == 0 || op == 7 || op == 8) {
      uint32_t left = ln;
      while (left) {
        if (mnum) {
          if (op == 8) MD_FAIL(E_MD_SPAN, r);
          const uint32_t t = mnum < (long long)left ? (uint32_t)mnum : left;
          const uint8_t* bad = (const uint8_t*)memchr(codes + q, 0xff, t);
          if (bad) MD_FAIL(E_N_MATCH, bad - codes);
          run += t; mnum -= t; q += (int32_t)t; r += (int32_t)t; left -= t;
        } else {
          if (!*c || *c == '^' || op == 7) MD_FAIL(E_MD_SPAN, r);
          const int rc_ = base_code(*c++);
          mnum = md_num(&c);
          if (codes[q] > 3) MD_FAIL(E_SUB_N, q);
          MD_FLUSH();
          ops[n++] = HM_MAKE_SUB(rc_ < 0 ? HM_BASE_N : (uint32_t)rc_, (uint32_t)codes[q]);
          q++; r++; left--;
        }
      }
    } else if (op == 1) {
      MD_FLUSH();
      ops[n++] = HM_MAKE_OP(HM_OP_INS, ln);
      q += (int32_t)ln;
    } else { /* D */
      if (mnum || *c != '^') MD_FAIL(E_MD_SPAN, r);
      const char* s0 = ++c;
      while (is_alpha(*c)) c++;
      if ((uint32_t)(c - s0) != ln) MD_FAIL(E_MD_SPAN, r);
      mnum = md_num(&c);
      MD_FLUSH();
      ops[n++] = HM_MAKE_OP(HM_OP_DEL, ln);
      r += (int32_t)ln;
    }
  }
  MD_FLUSH();
  if (mnum || *c) MD_FAIL(E_MD_SPAN, r);
#undef MD_FLUSH
#undef MD_FAIL
  *n_out = n; *q_out = q; *rspan_out = r;
  return 1;
}

/* phase B for one record: SEQ -> 2-bit, QUAL copy, cs -> ops (cslib.cs2lst grammar), CIGAR + MD -> ops (md_walk) or
 * CIGAR + reference -> ops (ref_walk, into the worker's scratch, then R->ext) with span and base checks */
static void decode_record(hm_bam* b, rec_t* R, uint8_t** codes_p, size_t* codes_cap, uint32_t** scratch, size_t* scratch_cap) {
  const uint8_t* r = R->rec;
  const uint32_t l_name = r[8], n_cig = r[12] | (r[13] << 8);
  const int32_t l_seq = R->l_seq;
  const uint8_t* seq4 = r + 32 + l_name + 4 * (size_t)n_cig;
  const uint8_t* qual = seq4 + ((size_t)l_seq + 1) / 2;
  if ((size_t)l_seq + 2 > *codes_cap) {
    size_t nc = (size_t)l_seq + 4096;
    uint8_t* np_ = (uint8_t*)realloc(*codes_p, nc);
    if (!np_) { R->err = E_CS_TOKEN; R->err_arg = -1; return; }
    *codes_p = np_; *codes_cap = nc;
  }
  uint8_t* codes = *codes_p;
  nib_to_codes_scalar(seq4, have_ssse3() ? nib_to_codes_simd(seq4, l_seq, codes) : 0, l_seq, codes);
  uint32_t* ops = b->ops + R->op_slot;
  uint32_t n_ops = 0;
  int32_t q = R->lead, rspan = 0;
  const char* cs = R->cs;
  const char* c = cs;
  const int by_ref = !cs && !R->md;
  if (by_ref) {
    const size_t need = 2 * (size_t)l_seq + n_cig + 2;
    if (need > *scratch_cap) {
      uint32_t* np_ = (uint32_t*)realloc(*scratch, need * sizeof(uint32_t));
      if (!np_) { R->err = E_NO_MEM; R->err_arg = (long)(need * sizeof(uint32_t)); return; }
      *scratch = np_; *scratch_cap = need;
    }
    ops = *scratch;
    if (!ref_walk(b, R, r + 32 + l_name, n_cig, codes, l_seq, ops, &n_ops, &q, &rspan)) return;
  } else if (!cs && !md_walk(R, r + 32 + l_name, n_cig, codes, l_seq, ops, &n_ops, &q, &rspan)) return;
  while (cs && *c) {
    if (*c == ':') {
      long n = 0; c++;
      if (*c < '0' || *c > '9') { R->err = E_CS_TOKEN; R->err_arg = (long)(c - cs); return; }
      while (*c >= '0' && *c <= '9') { n = n * 10 + (*c++ - '0'); if (n > l_seq) { R->err = E_CS_PAST; R->err_arg = n; return; } }
      if (q + n > l_seq) { R->err = E_CS_PAST; R->err_arg = q + n; return; }
      if (n) { const uint8_t* bad = (const uint8_t*)memchr(codes + q, 0xff, (size_t)n); if (bad) { R->err = E_N_MATCH; R->err_arg = (long)(bad - codes); return; } }
      if (n) ops[n_ops++] = HM_MAKE_OP(HM_OP_MATCH, n);
      q += (int32_t)n; rspan += (int32_t)n;
    } else if (*c == '=') {
      long n = 0; c++;
      while ((c[n] >= 'A' && c[n] <= 'Z') || (c[n] >= 'a' && c[n] <= 'z')) n++;
      if (n == 0 || q + n > l_seq) { R->err = E_CS_TOKEN; R->err_arg = (long)(c - cs); return; }
      for (long k = 0; k < n; k++) {
        int bc = base_code(c[k]);
        if (bc < 0 || codes[q + k] != (uint8_t)bc) { R->err = E_CS_LONG; R->err_arg = q + k; return; }
      }
      ops[n_ops++] = HM_MAKE_OP(HM_OP_MATCH, n);
      c += n; q += (int32_t)n; rspan += (int32_t)n;
    } else if (*c == '*') {
      if (!c[1] || !c[2]) { R->err = E_CS_TOKEN; R->err_arg = (long)(c - cs); return; }
      int rc_ = base_code(c[1]), ac = base_code(c[2]);
      if (ac < 0) { R->err = E_SUB_N; R->err_arg = q; return; }
      ops[n_ops++] = HM_MAKE_SUB(rc_ < 0 ? HM_BASE_N : (uint32_t)rc_, (uint32_t)ac);
      c += 3; q += 1; rspan += 1;
    } else if (*c == '+' || *c == '-') {
      int ins = *c == '+';
      long n = 0; c++;
      while ((c[n] >= 'A' && c[n] <= 'Z') || (c[n] >= 'a' && c[n] <= 'z')) n++;
      if (n == 0) { R->err = E_CS_TOKEN; R->err_arg = (long)(c - cs); return; }
      ops[n_ops++] = HM_MAKE_OP(ins ? HM_OP_INS : HM_OP_DEL, n);
      c += n;
      if (ins) q += (int32_t)n; else rspan += (int32_t)n;
    } else { R->err = E_CS_TOKEN; R->err_arg = (long)(c - cs); return; }
  }
  if (rspan != R->ref_span) { R->err = E_SPAN_REF; R->err_arg = rspan; return; }
  if (q - R->lead != l_seq - R->trail - R->lead) { R->err = E_SPAN_QRY; R->err_arg = q - R->lead; return; }
  if (by_ref) {
    R->ext = (uint32_t*)malloc((n_ops ? n_ops : 1) * sizeof(uint32_t));
    if (!R->ext) { R->err = E_NO_MEM; R->err_arg = (long)((n_ops ? n_ops : 1) * sizeof(uint32_t)); return; }
    memcpy(R->ext, ops, (size_t)n_ops * sizeof(uint32_t));
  }
  R->n_ops = n_ops; R->rspan = rspan;
  const size_t sb = ((size_t)l_seq + 3) / 4, sb16 = (sb + 15) & ~(size_t)15, qb16 = ((size_t)l_seq + 15) & ~(size_t)15;
  if (!b->no_seq) {
    uint8_t* dst = b->seq + R->seq_off;
    pack_codes_scalar(codes, have_ssse3() ? pack_codes_simd(codes, l_seq, dst) : 0, l_seq, dst);
    memset(dst + sb, 0, sb16 - sb);
  }
  if (!b->compact_bq) {
    memcpy(b->bq + R->bq_off, qual, (size_t)l_seq);
    memset(b->bq + R->bq_off + l_seq, 0, qb16 - (size_t)l_seq);
  } else {
    /* hm_bq_compact: one bit per byte of the expanded stream (set: the modal quality; padding bits clear), the other
     * qualities in base order.  16 qualities per step. */
    uint8_t* m = b->qmask + (R->bq_off >> 3);
    uint8_t* e = b->qexc + R->exc_slot;
    const uint8_t modal = (uint8_t)b->modal;
    uint32_t ne = 0;
    int32_t i = 0;
#if defined(__SSE2__)
    const __m128i vm = _mm_set1_epi8((char)modal);
    for (; i + 16 <= l_seq; i += 16) {
      const uint32_t eq = (uint32_t)_mm_movemask_epi8(_mm_cmpeq_epi8(_mm_loadu_si128((const __m128i*)(qual + i)), vm));
      m[i >> 3] = (uint8_t)eq; m[(i >> 3) + 1] = (uint8_t)(eq >> 8);
      uint32_t z = ~eq & 0xffffu;
      while (z) { const int k = __builtin_ctz(z); z &= z - 1; e[ne++] = qual[i + k]; }
    }
#endif
    for (; i < l_seq; i += 16) { /* the last, partial group (every group without SSE2) */
      uint32_t eq = 0;
      const int32_t lim = l_seq - i < 16 ? l_seq - i : 16;
      for (int32_t k = 0; k < lim; k++) { if (qual[i + k] == modal) eq |= 1u << k; else e[ne++] = qual[i + k]; }
      m[i >> 3] = (uint8_t)eq; m[(i >> 3) + 1] = (uint8_t)(eq >> 8);
    }
    R->n_exc = ne;
  }
}

static void* decode_worker(void* arg) {
  decode_job_t* j = (decode_job_t*)arg;
  uint8_t* codes = NULL; size_t cap = 0;
  uint32_t* scratch = NULL; size_t scap = 0;
  for (;;) {
    pthread_mutex_lock(&j->mu);
    size_t i0 = j->next;
    j->next += 64;
    pthread_mutex_unlock(&j->mu);
    if (i0 >= j->n) break;
    for (size_t i = i0; i < i0 + 64 && i < j->n; i++) decode_record(j->b, &j->recs[i], &codes, &cap, &scratch, &scap);
  }
  free(codes); free(scratch);
  return NULL;
}

int hm_bam_set_option(hm_bam* b, int option, int value) {
  if (!b) return HM_ERR_ARG;
  if (option == HM_BAM_OPT_NO_SEQ) { b->no_seq = value != 0; return HM_OK; }
  if (option == HM_BAM_OPT_COMPACT_BQ) { b->compact_bq = value != 0; return HM_OK; }
  if (option == HM_BAM_OPT_BUFFER_SET) {
    if (value != 0 && value != 1) return fail(b, "buffer set must be 0 or 1%s (%ld)", NULL, (long)value);
    if (value != b->cur_set) { swap_bufset(b); b->cur_set = value; }
    return HM_OK;
  }
  return fail(b, "unknown option%s (%ld)", NULL, (long)option);
}

int hm_bam_read_batch(hm_bam* b, int rid, int32_t start, int32_t end, int threads, hm_read_batch* out) {
  if (!b || !out) return HM_ERR_ARG;
  if (rid < 0 || rid >= b->n_ref) return fail(b, "invalid contig index%s %ld", NULL, rid);
  if (start < 0) start = 0;
  if (end > b->refs[rid].len) end = b->refs[rid].len;
  size_t n_reads = 0, n_seq = 0, n_bq = 0, n_ops = 0;
  uint64_t n_exc = 0;
  memset(out, 0, sizeof(*out));
  b->n_qexc = 0;
  const uint64_t voff = seek_voff(b, rid, start);
  if (!voff) goto finish; /* no reads on this contig */
  {
    stream_t s;
    memset(&s, 0, sizeof(s));
    s.b = b; s.threads = threads;
    { /* first read sized for the region (about 8 compressed bytes per reference position at 30x), so that a large
         region keeps every inflate thread busy from the start */
      const uint64_t guess = (uint64_t)(end > start ? end - start : 0) * 8u;
      s.span = guess < (1u << 20) ? (1u << 20) : (guess > (64u << 20) ? (64u << 20) : (size_t)guess);
    }
    if (stream_seek(&s, voff) < 0) { free(s.buf); return fail(b, "cannot read BGZF blocks of %s (%ld)", b->path, 0); }
    rec_t* recs = NULL; size_t recs_cap = 0;
    int rc = HM_OK, done = 0;
    const int nt = threads < 1 ? 1 : (threads > 64 ? 64 : threads);
    while (!done && !rc) {
      /* phase A (serial): every complete record now in the buffer — select, validate what needs file order,
       * intern the query name, assign output space */
      int st = stream_need(&s, 4);
      if (st == 1) break;
      if (st < 0) { rc = fail(b, "truncated BAM %s (%ld)", b->path, 0); break; }
      {
        uint32_t bs0 = rd32(s.buf + s.pos);
        if (stream_need(&s, 4 + (size_t)bs0)) { rc = fail(b, REC_ERR[E_TRUNC_REC], b->path, 0); break; }
      }
      double tA = now_s();
      size_t nsel = 0, seg_ops = 0, seg_exc = 0, seg_ref = 0;
      const size_t first_read = n_reads;
      while (s.len - s.pos >= 4) {
        uint32_t bs = rd32(s.buf + s.pos);
        if (s.len - s.pos < 4 + (size_t)bs) break; /* partial record: next fill */
        const uint8_t* r = s.buf + s.pos + 4;
        s.pos += 4 + (size_t)bs;
        int32_t ref_id = (int32_t)rd32(r), pos = (int32_t)rd32(r + 4);
        if (ref_id != rid) { if (ref_id > rid || ref_id < 0) { done = 1; break; } continue; }
        if (pos >= end) { done = 1; break; }
        if (bs < 32) { rc = fail(b, REC_ERR[E_BLOCK_SIZE], b->path, (long)bs); break; }
        uint32_t l_name = r[8], mapq = r[9], n_cig = r[12] | (r[13] << 8), flag = r[14] | (r[15] << 8);
        int32_t l_seq = (int32_t)rd32(r + 16);
        /* the fixed part, name, CIGAR, SEQ and QUAL must lie inside the record before any of them is touched */
        if (l_seq < 0 || l_name == 0 || 32 + (uint64_t)l_name + 4 * (uint64_t)n_cig + ((uint64_t)l_seq + 1) / 2 + (uint64_t)l_seq > (uint64_t)bs ||
            r[32 + l_name - 1] != 0) {
          rc = fail(b, REC_ERR[E_FIELDS], b->path, (long)bs);
          break;
        }
        const char* qname = (const char*)(r + 32);
        const uint8_t* cig = r + 32 + l_name;
        int32_t ref_span = 0, lead = 0, trail = 0;
        for (uint32_t k = 0; k < n_cig; k++) {
          uint32_t c = rd32(cig + 4 * k), op = c & 15, ln = c >> 4;
          if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) ref_span += (int32_t)ln;
        }
        for (uint32_t k = 0; k < n_cig; k++) { uint32_t c = rd32(cig + 4 * k), op = c & 15; if (op == 4) lead += (int32_t)(c >> 4); else if (op != 5) break; }
        for (uint32_t k = n_cig; k-- > 0;) { uint32_t c = rd32(cig + 4 * k), op = c & 15; if (op == 4) trail += (int32_t)(c >> 4); else if (op != 5) break; }
        int32_t rend = pos + (ref_span > 0 ? ref_span : 1);
        if (rend <= start) continue;
        if (flag & 0x100) continue; /* secondary: bamlib.py:17 */
        const uint8_t* seq4 = cig + 4 * (size_t)n_cig;
        const uint8_t* qual = seq4 + ((size_t)l_seq + 1) / 2;
        const uint8_t* tag = qual + (l_seq > 0 ? l_seq : 0);
        const uint8_t* rec_end = r + bs;
        const char* cs = NULL;
        const char* md = NULL;
        while (tag + 3 <= rec_end) {
          char ty = (char)tag[2];
          const uint8_t* v = tag + 3;
          const size_t left = (size_t)(rec_end - v);
          size_t adv;
          if (ty == 'Z' || ty == 'H') {
            const void* z = memchr(v, 0, left); /* the string must end inside the record */
            if (!z) { rc = fail(b, REC_ERR[E_TAG_UNTERM], qname, (long)ty); break; }
            adv = (size_t)((const uint8_t*)z - v) + 1;
            if (tag[0] == 'c' && tag[1] == 's' && ty == 'Z') cs = (const char*)v;
            if (tag[0] == 'M' && tag[1] == 'D' && ty == 'Z') md = (const char*)v;
          }
          else if (ty == 'A' || ty == 'c' || ty == 'C') adv = 1;
          else if (ty == 's' || ty == 'S') adv = 2;
          else if (ty == 'i' || ty == 'I' || ty == 'f') adv = 4;
          else if (ty == 'B') {
            if (left < 5) { rc = fail(b, REC_ERR[E_TAG_B], qname, (long)left); break; }
            const size_t esz = b_elem_size((char)v[0]);
            if (!esz) { rc = fail(b, REC_ERR[E_TAG_B], qname, (long)v[0]); break; }
            adv = 5 + (size_t)rd32(v + 1) * esz;
          }
          else { rc = fail(b, REC_ERR[E_TAG_TYPE], qname, ty); break; }
          if (adv > left) { rc = fail(b, REC_ERR[E_TAG_PAST], qname, (long)adv); break; }
          tag = v + adv;
        }
        if (rc) break;
        /* cs when it is there, else CIGAR + MD, else CIGAR + the reference when the caller set this contig's */
        const int by_ref = !cs && !md && b->ref_seq && b->ref_rid == rid;
        if (!cs && !md && !by_ref) { rc = fail(b, REC_ERR[E_NO_CS], qname, 0); break; }
        /* hard clips: pysam's query_sequence and query_alignment_start leave them out (SEQ holds no hard-clipped base),
         * so cs2tuple indexes consistently and the reference processes such records (minimap2 writes them for
         * supplementary alignments without -Y); lead / trail above count soft clips only */
        if (l_seq <= 0 || qual[0] == 0xff) { rc = fail(b, REC_ERR[E_NO_QUAL], qname, 0); break; }
        if (nsel == recs_cap) {
          size_t nc = recs_cap ? recs_cap * 2 : 8192;
          rec_t* nr = (rec_t*)realloc(recs, nc * sizeof(rec_t));
          if (!nr) { rc = fail(b, "out of memory%s (%ld)", NULL, (long)nc); break; }
          recs = nr; recs_cap = nc;
        }
        if (n_reads + 1 > b->cap_reads) {
          size_t cr = b->cap_reads ? b->cap_reads + b->cap_reads / 2 + 1024 : 4096;
#define RE(ptr, type) do { type* np_ = (type*)realloc(ptr, cr * sizeof(type)); if (!np_) rc = fail(b, "out of memory%s (%ld)", NULL, (long)cr); else ptr = np_; } while (0)
          RE(b->tstart, int32_t); RE(b->tend, int32_t); RE(b->qstart, int32_t); RE(b->qlen, int32_t); RE(b->mapq, uint8_t);
          RE(b->flags, uint8_t); RE(b->qname_id, uint32_t); RE(b->n_ops, uint32_t); RE(b->seq_off, uint64_t);
          RE(b->bq_off, uint64_t); RE(b->op_off, uint64_t);
#undef RE
          if (rc) break;
          b->cap_reads = cr;
        }
        int64_t id = qt_get(&b->qt, qname, strlen(qname));
        if (id < 0) { rc = fail(b, "out of memory%s (%ld)", NULL, 0); break; }
        const size_t sb = ((size_t)l_seq + 3) / 4, sb16 = (sb + 15) & ~(size_t)15, qb16 = ((size_t)l_seq + 15) & ~(size_t)15;
        rec_t* R = &recs[nsel++];
        R->rec = r; R->cs = cs; R->md = cs ? NULL : md; R->ext = NULL; R->pos = pos; R->l_seq = l_seq; R->lead = lead; R->trail = trail; R->ref_span = ref_span;
        R->seq_off = n_seq; R->bq_off = n_bq; R->op_slot = n_ops + seg_ops; R->n_ops = 0; R->rspan = 0; R->err = 0; R->err_arg = 0;
        R->exc_slot = (size_t)n_exc + seg_exc; R->n_exc = 0;
        if (b->compact_bq) {
          if (!b->modal) { /* the handle's modal quality: the most frequent one of the first record it compacts */
            uint32_t hist[256]; memset(hist, 0, sizeof(hist));
            for (int32_t k = 0; k < l_seq; k++) hist[qual[k]]++;
            int mo = 1;
            for (int v_ = 1; v_ < 255; v_++) if (hist[v_] > hist[mo]) mo = v_;
            b->modal = mo;
          }
          seg_exc += (size_t)l_seq;
        }
        b->tstart[n_reads] = pos; b->qstart[n_reads] = lead; b->qlen[n_reads] = l_seq;
        b->mapq[n_reads] = (uint8_t)mapq; b->flags[n_reads] = 0; b->qname_id[n_reads] = (uint32_t)id;
        b->seq_off[n_reads] = n_seq; b->bq_off[n_reads] = n_bq;
        if (!b->no_seq) n_seq += sb16;
        /* ops of CIGAR + MD: SUBs <= MD letters, INS + DEL <= CIGAR ops, match runs <= the other ops + 1; CIGAR +
         * reference: no slot (R->ext) */
        n_bq += qb16; n_reads++;
        if (by_ref) seg_ref++;
        else seg_ops += cs ? strlen(cs) / 2 + 2 : 2 * (strlen(md) + n_cig) + 2;
      }
      if (rc) break;
      if (nsel) {
        if (!b->no_seq) GROW(b->seq, b->cap_seq, n_seq + 16, uint8_t);
        if (!b->compact_bq) GROW(b->bq, b->cap_bq, n_bq + 16, uint8_t);
        else {
          GROW(b->qmask, b->cap_qmask, (n_bq >> 3) + 16, uint8_t);
          GROW(b->qexc, b->cap_qexc, (size_t)n_exc + seg_exc + 32, uint8_t);
          GROW(b->qexc_off, b->cap_qexc_off, n_reads + 2, uint64_t);
        }
        GROW(b->ops, b->cap_ops, n_ops + seg_ops + 4, uint32_t);
        g_phase[4] += now_s() - tA; tA = now_s();
        /* phase B (parallel): bases, qualities, cs -> ops */
        decode_job_t job;
        memset(&job, 0, sizeof(job));
        job.b = b; job.recs = recs; job.n = nsel;
        pthread_mutex_init(&job.mu, NULL);
        int use = nt;
        if ((size_t)use > (nsel + 63) / 64) use = (int)((nsel + 63) / 64);
        pthread_t th[64];
        for (int t = 1; t < use; t++) pthread_create(&th[t], NULL, decode_worker, &job);
        decode_worker(&job);
        for (int t = 1; t < use; t++) pthread_join(th[t], NULL);
        pthread_mutex_destroy(&job.mu);
        g_phase[5] += now_s() - tA; tA = now_s();
        /* serial tail: first error in file order, op compaction.  Ops of CIGAR + reference records (R->ext) are counted
         * only by their decode, so with any of them the segment's ops are gathered past the slots and moved down. */
        size_t gather = 0;
        const size_t ops0 = n_ops;
        if (seg_ref) {
          size_t tot = 0;
          for (size_t i = 0; i < nsel; i++) tot += recs[i].n_ops;
          gather = n_ops + seg_ops;
          if (gather + tot + 4 > b->cap_ops) {
            uint32_t* np_ = (uint32_t*)realloc(b->ops, (gather + tot + 4) * sizeof(uint32_t));
            if (!np_) rc = fail(b, "out of memory%s (%ld)", NULL, (long)(gather + tot + 4));
            else { b->ops = np_; b->cap_ops = gather + tot + 4; }
          }
        }
        for (size_t i = 0; i < nsel && !rc; i++) {
          rec_t* R = &recs[i];
          if (R->err) { rc = fail(b, REC_ERR[R->err], (const char*)(R->rec + 32), R->err_arg); break; }
          const size_t rd = first_read + i;
          if (seg_ref) memcpy(b->ops + gather + (n_ops - ops0), R->ext ? R->ext : b->ops + R->op_slot, (size_t)R->n_ops * sizeof(uint32_t));
          else if (R->op_slot != n_ops) memmove(b->ops + n_ops, b->ops + R->op_slot, (size_t)R->n_ops * sizeof(uint32_t));
          b->op_off[rd] = n_ops; b->n_ops[rd] = R->n_ops; b->tend[rd] = R->pos + R->rspan;
          n_ops += R->n_ops;
          if (b->compact_bq) {
            if (R->exc_slot != n_exc) memmove(b->qexc + n_exc, b->qexc + R->exc_slot, (size_t)R->n_exc);
            b->qexc_off[rd] = n_exc;
            n_exc += R->n_exc;
          }
        }
        if (seg_ref && !rc) memmove(b->ops + ops0, b->ops + gather, (n_ops - ops0) * sizeof(uint32_t));
        if (seg_ref) for (size_t i = 0; i < nsel; i++) { free(recs[i].ext); recs[i].ext = NULL; }
      }
    }
    if (getenv("HIMUT_B200_DECODE_TIMING"))
      fprintf(stderr, "[decode timing] read %.3f walk %.3f inflate %.3f free %.3f | scan+alloc %.3f decode %.3f s\n", g_phase[0], g_phase[1], g_phase[2], g_phase[3], g_phase[4], g_phase[5]);
    memset(g_phase, 0, sizeof(g_phase));
    free(recs); free(s.buf);
    if (rc) return rc;
  }
finish:
  if (n_seq == 0 && !b->no_seq) { GROW(b->seq, b->cap_seq, 16, uint8_t); memset(b->seq, 0, 16); n_seq = 16; }
  if (n_bq == 0) {
    if (!b->compact_bq) { GROW(b->bq, b->cap_bq, 16, uint8_t); memset(b->bq, 0, 16); }
    else { GROW(b->qmask, b->cap_qmask, 16, uint8_t); memset(b->qmask, 0, 16); }
    n_bq = 16;
  }
  if (b->compact_bq) {
    GROW(b->qexc_off, b->cap_qexc_off, n_reads + 2, uint64_t);
    GROW(b->qexc, b->cap_qexc, (size_t)n_exc + 32, uint8_t);
    b->qexc_off[n_reads] = n_exc;
    memset(b->qexc + n_exc, 0, 32); /* the expansion kernel may read a few bytes past the last exception */
    b->n_qexc = n_exc;
    if (!b->modal) b->modal = 93;
  }
  out->n_reads = n_reads;
  out->tstart = b->tstart; out->tend = b->tend; out->qstart = b->qstart; out->qlen = b->qlen; out->mapq = b->mapq;
  out->flags = b->flags; out->qname_id = b->qname_id; out->seq_off = b->seq_off; out->bq_off = b->bq_off;
  out->op_off = b->op_off; out->n_ops = b->n_ops; out->seq = b->seq; out->seq_bytes = n_seq; out->bq = b->bq;
  out->bq_bytes = n_bq; out->ops = b->ops; out->n_ops_total = n_ops;
  if (b->no_seq) { out->seq = NULL; out->seq_off = NULL; out->seq_bytes = 0; } /* himut_b200.h: a batch without a base stream */
  if (b->compact_bq) out->bq = NULL; /* the qualities are in hm_bam_last_compact; bq_off / bq_bytes describe the expanded layout */
  b->batch = *out;
  return HM_OK;
}

int hm_bam_last_compact(hm_bam* b, hm_bq_compact* out) {
  if (!b || !out) return HM_ERR_ARG;
  if (!b->compact_bq || !b->qmask) return fail(b, "the last batch was not decoded with HM_BAM_OPT_COMPACT_BQ%s (%ld)", NULL, 0);
  memset(out, 0, sizeof(*out));
  out->mask = b->qmask; out->mask_bytes = b->batch.bq_bytes >> 3;
  out->exc = b->qexc; out->exc_bytes = b->n_qexc; out->exc_off = b->qexc_off;
  out->modal = (uint8_t)b->modal;
  return HM_OK;
}

/* ------------------------------------------------------------------ region plan for the device decoder */
/* the BGZF header at coff: 0 and *blk filled, 1 end of file, -1 not a BGZF block */
static int block_at(hm_bam* b, uint64_t coff, blk_t* blk, uint32_t* crc) {
  if (!b->map) {
    const int st = read_block_header(b->f, coff, blk);
    if (st) return st;
    uint8_t t[4];
    if (fseeko(b->f, (off_t)(coff + blk->csize - 8), SEEK_SET) || fread(t, 1, 4, b->f) != 4) return -1;
    *crc = rd32(t);
    return 0;
  }
  if (coff >= b->map_len) return 1;
  const uint8_t* h = b->map + coff;
  if (b->map_len - coff < 18 || h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4)) return -1;
  const uint16_t xlen = (uint16_t)(h[10] | (h[11] << 8));
  if (coff + 12 + xlen > b->map_len) return -1;
  int bsize = -1;
  for (int q = 0; q + 4 <= xlen;) {
    const int slen = h[12 + q + 2] | (h[12 + q + 3] << 8);
    if (h[12 + q] == 66 && h[12 + q + 1] == 67 && slen == 2) bsize = h[12 + q + 4] | (h[12 + q + 5] << 8);
    q += 4 + slen;
  }
  if (bsize < 0 || (size_t)bsize + 1 < 12u + xlen + 8u || coff + (uint64_t)bsize + 1 > b->map_len) return -1;
  blk->coff = coff; blk->csize = (uint32_t)bsize + 1;
  blk->usize = rd32(h + blk->csize - 4);
  *crc = rd32(h + blk->csize - 8);
  return 0;
}

static int plan_range(hm_bam* b, uint64_t v_lo, uint64_t v_hi, const uint64_t* ventry, size_t n_ventry, hm_bgzf_plan* out);

int hm_bam_region_plan(hm_bam* b, int rid, int32_t start, int32_t end, hm_bgzf_plan* out) {
  if (!b || !out) return HM_ERR_ARG;
  if (rid < 0 || rid >= b->n_ref) return fail(b, "invalid contig index%s %ld", NULL, rid);
  memset(out, 0, sizeof(*out));
  out->path = b->path;
  if (start < 0) start = 0;
  if (end > b->refs[rid].len) end = b->refs[rid].len;
  uint64_t v_lo = b->first_record, v_hi = UINT64_MAX; /* UINT64_MAX: to the end of the file */
  uint64_t* ventry = NULL; /* virtual offsets of the later entry points */
  size_t n_ventry = 0;
  if (b->index_kind) {
    const bam_ref_t* R = &b->refs[rid];
    const int ms = b->min_shift, depth = b->depth;
    /* where hm_bam_read_batch seeks to */
    v_lo = seek_voff(b, rid, start);
    if (!v_lo) return HM_OK; /* no reads on this contig: an empty plan */
    /* every record that overlaps the region (hm_bam_read_batch's rule: pos < end, reference end > start) lies in a
     * chunk of a bin that overlaps [min(start, end), max(start, end) + 1): the range ends at their largest end.  The
     * large bins overlap every region and their chunks reach to the far end of the contig, so the range also ends at
     * the first chunk of any bin that starts at or past `end`: every record there has pos >= end, where
     * hm_bam_read_batch stops, and it is a record start. */
    const int64_t rb = start < end ? start : end, re = (int64_t)(start > end ? start : end) + 1; /* end may be 2^31 - 1 */
    v_hi = 0;
    for (int32_t k = 0; k < R->n_bin; k++) {
      const int64_t bs = bin_start(R->bins[k].id, ms, depth);
      if (bs < re && bs + bin_size(R->bins[k].id, ms, depth) > rb && R->bins[k].end > v_hi) v_hi = R->bins[k].end;
    }
    for (int32_t k = 0; k < R->n_bin; k++)
      if (bin_start(R->bins[k].id, ms, depth) >= (int64_t)end && R->bins[k].beg < v_hi) v_hi = R->bins[k].beg;
    if (v_hi <= v_lo) return HM_OK; /* no record overlaps the region */
    if (b->index_kind == HM_BAM_INDEX_BAI) {
      /* the linear-index entries of the windows the region covers */
      int32_t w0 = start >> 14;
      if (w0 >= R->n_lin) w0 = R->n_lin - 1;
      const int32_t w_last = (int32_t)((re - 1) >> 14) < R->n_lin - 1 ? (int32_t)((re - 1) >> 14) : R->n_lin - 1;
      if (w_last > w0) {
        ventry = (uint64_t*)malloc((size_t)(w_last - w0) * sizeof(uint64_t));
        if (!ventry) return fail(b, "out of memory%s (%ld)", NULL, 0);
      }
      for (int32_t k = w0 + 1; k <= w_last; k++)
        if (R->lin[k] > v_lo && R->lin[k] < v_hi && (!n_ventry || R->lin[k] > ventry[n_ventry - 1])) ventry[n_ventry++] = R->lin[k];
    } else {
      /* the loffsets of the bins of any level that start inside the region: each is a record start.  A read that
       * crosses a window boundary goes to a larger bin, so the leaf bins alone would leave long serial segments. */
      ventry = (uint64_t*)malloc(((size_t)R->n_bin + 1) * sizeof(uint64_t));
      if (!ventry) return fail(b, "out of memory%s (%ld)", NULL, 0);
      for (int32_t k = 0; k < R->n_bin; k++) {
        const int64_t bs = bin_start(R->bins[k].id, ms, depth);
        const uint64_t v = R->bins[k].loff;
        if (bs >= rb && bs < re && v > v_lo && v < v_hi) ventry[n_ventry++] = v;
      }
      qsort(ventry, n_ventry, sizeof(uint64_t), cmp_u64);
      size_t m = 0;
      for (size_t k = 0; k < n_ventry; k++) if (!m || ventry[k] != ventry[m - 1]) ventry[m++] = ventry[k];
      n_ventry = m;
    }
  }
  const int rc = plan_range(b, v_lo, v_hi, ventry, n_ventry, out);
  free(ventry);
  return rc;
}

/* hm_bam_region_plan from virtual offsets: the first entry point, the end of the range (UINT64_MAX: the end of the
 * file) and the later entry points, ascending */
static int plan_range(hm_bam* b, uint64_t v_lo, uint64_t v_hi, const uint64_t* ventry, size_t n_ventry, hm_bgzf_plan* out) {
  /* the block table of the compressed range, by the header walk stream_fill does */
  const uint64_t c_lo = v_lo >> 16;
  size_t nb = 0;
  uint64_t usum = 0, coff = c_lo;
  for (;;) {
    if (v_hi != UINT64_MAX && (coff > (v_hi >> 16) || (coff == (v_hi >> 16) && (v_hi & 0xffff) == 0))) break;
    blk_t blk;
    uint32_t crc = 0;
    const int st = block_at(b, coff, &blk, &crc);
    if (st == 1 && v_hi == UINT64_MAX) break;
    if (st) return fail(b, "cannot read BGZF blocks of %s (%ld)", b->path, (long)coff);
    if (nb + 2 > b->cap_plan_blocks) {
      const size_t nc = b->cap_plan_blocks ? 2 * b->cap_plan_blocks : 4096;
#define RP(ptr, type) do { type* np_ = (type*)realloc(ptr, nc * sizeof(type)); if (!np_) return fail(b, "out of memory%s (%ld)", NULL, (long)nc); ptr = np_; } while (0)
      RP(b->p_coff, uint64_t); RP(b->p_uoff, uint64_t); RP(b->p_csize, uint32_t); RP(b->p_isize, uint32_t); RP(b->p_crc, uint32_t);
#undef RP
      b->cap_plan_blocks = nc;
    }
    b->p_coff[nb] = coff - c_lo; b->p_csize[nb] = blk.csize; b->p_isize[nb] = blk.usize; b->p_crc[nb] = crc; b->p_uoff[nb] = usum;
    if (blk.usize > 65536) return fail(b, "cannot read BGZF blocks of %s (%ld)", b->path, (long)coff);
    usum += blk.usize; coff += blk.csize; nb++;
  }
  if (nb == 0) return HM_OK;
  b->p_coff[nb] = coff - c_lo;
  b->p_uoff[nb] = usum;
  /* virtual offset -> offset in the inflated range; an in-block offset equal to ISIZE is the next block's start */
#define V2U(v, dst)                                                                                              \
  do {                                                                                                           \
    const uint64_t c_ = ((v) >> 16) - c_lo;                                                                      \
    size_t lo_ = 0, hi_ = nb;                                                                                    \
    while (lo_ < hi_) { const size_t m_ = (lo_ + hi_) / 2; if (b->p_coff[m_] < c_) lo_ = m_ + 1; else hi_ = m_; } \
    if (b->p_coff[lo_] != c_ || (lo_ < nb && ((v) & 0xffff) > b->p_isize[lo_]) || (lo_ == nb && ((v) & 0xffff)))  \
      return fail(b, b->index_kind == HM_BAM_INDEX_CSI ? "CSI virtual offset outside the BGZF blocks of %s (%ld)"  \
                                                        : "BAI virtual offset outside the BGZF blocks of %s (%ld)", b->path, \
                  (long)((v) >> 16));                                                                            \
    (dst) = b->p_uoff[lo_] + ((v) & 0xffff);                                                                     \
  } while (0)
  uint64_t u_end = usum;
  if (v_hi != UINT64_MAX) V2U(v_hi, u_end);
  if (n_ventry + 1 > b->cap_plan_entry) {
    uint64_t* np_ = (uint64_t*)realloc(b->p_entry, (n_ventry + 1) * sizeof(uint64_t));
    if (!np_) return fail(b, "out of memory%s (%ld)", NULL, 0);
    b->p_entry = np_; b->cap_plan_entry = n_ventry + 1;
  }
  size_t ne = 0;
  V2U(v_lo, b->p_entry[ne]);
  ne++;
  for (size_t k = 0; k < n_ventry; k++) {
    uint64_t u;
    V2U(ventry[k], u);
    if (u > b->p_entry[ne - 1] && u < u_end) b->p_entry[ne++] = u;
  }
#undef V2U
  if (b->map) out->comp = b->map + c_lo;
  else {
    if (coff - c_lo > b->cap_p_comp) {
      uint8_t* np_ = (uint8_t*)realloc(b->p_comp, coff - c_lo);
      if (!np_) return fail(b, "out of memory%s (%ld)", NULL, 0);
      b->p_comp = np_; b->cap_p_comp = coff - c_lo;
    }
    if (fseeko(b->f, (off_t)c_lo, SEEK_SET) || fread(b->p_comp, 1, coff - c_lo, b->f) != coff - c_lo)
      return fail(b, "cannot read BGZF blocks of %s (%ld)", b->path, (long)c_lo);
    out->comp = b->p_comp;
  }
  out->comp_bytes = coff - c_lo;
  out->n_blocks = nb;
  out->blk_coff = b->p_coff; out->blk_csize = b->p_csize; out->blk_isize = b->p_isize; out->blk_uoff = b->p_uoff; out->blk_crc = b->p_crc;
  out->entry = b->p_entry; out->n_entry = ne;
  out->walk_end = u_end;
  return HM_OK;
}

int hm_bam_intern_qnames(hm_bam* b, const char* blob, const uint64_t* off, size_t n, uint32_t* ids) {
  if (!b || (n && (!blob || !off || !ids))) return HM_ERR_ARG;
  for (size_t i = 0; i < n; i++) {
    const char* s = blob + off[i];
    const int64_t id = qt_get(&b->qt, s, strlen(s));
    if (id < 0) return fail(b, "out of memory%s (%ld)", NULL, 0);
    ids[i] = (uint32_t)id;
  }
  return HM_OK;
}

/* ------------------------------------------------------------------ pre-pass: read lengths of a window */
/* bamlib.get_thresholds (src/himut/bamlib.py:137-178) fetches 100 random 100 kb windows per contig and keeps
 * len(query_sequence) of every record with mapping_quality > 0 and tp:A:P (secondary / supplementary records
 * included, as pysam's fetch returns them).  Only the fixed part of each record, its CIGAR and the tp tag are
 * looked at here: no base / quality unpacking, no cs parsing.  Lengths come back in fetch order. */
int hm_bam_window_qlens(hm_bam* b, int rid, int32_t start, int32_t end, int threads, int32_t* out, size_t cap, size_t* n_out) {
  if (!b || !n_out) return HM_ERR_ARG;
  *n_out = 0;
  if (rid < 0 || rid >= b->n_ref) return fail(b, "invalid contig index%s %ld", NULL, rid);
  if (start < 0) start = 0;
  if (end > b->refs[rid].len) end = b->refs[rid].len;
  if (start >= end) return HM_OK;
  const uint64_t voff = seek_voff(b, rid, start);
  if (!voff) return HM_OK;
  stream_t s;
  memset(&s, 0, sizeof(s));
  s.b = b; s.threads = threads;
  s.span = 1u << 18; /* windows are small: start with 256 KB of compressed data */
  if (stream_seek(&s, voff) < 0) { free(s.buf); return fail(b, "cannot read BGZF blocks of %s (%ld)", b->path, 0); }
  int rc = HM_OK;
  size_t n = 0;
  for (;;) {
    int st = stream_need(&s, 4);
    if (st == 1) break;
    if (st < 0) { rc = fail(b, "truncated BAM %s (%ld)", b->path, 0); break; }
    uint32_t bs = rd32(s.buf + s.pos);
    if (stream_need(&s, 4 + (size_t)bs)) { rc = fail(b, REC_ERR[E_TRUNC_REC], b->path, 0); break; }
    const uint8_t* r = s.buf + s.pos + 4;
    s.pos += 4 + (size_t)bs;
    int32_t ref_id = (int32_t)rd32(r), pos = (int32_t)rd32(r + 4);
    if (ref_id != rid) { if (ref_id > rid || ref_id < 0) break; continue; }
    if (pos >= end) break;
    if (bs < 32) { rc = fail(b, REC_ERR[E_BLOCK_SIZE], b->path, (long)bs); break; }
    uint32_t l_name = r[8], mapq = r[9], n_cig = r[12] | (r[13] << 8);
    int32_t l_seq = (int32_t)rd32(r + 16);
    if (l_seq < 0 || l_name == 0 || 32 + (uint64_t)l_name + 4 * (uint64_t)n_cig + ((uint64_t)l_seq + 1) / 2 + (uint64_t)l_seq > (uint64_t)bs ||
        r[32 + l_name - 1] != 0) {
      rc = fail(b, REC_ERR[E_FIELDS], b->path, (long)bs);
      break;
    }
    const uint8_t* cig = r + 32 + l_name;
    int32_t ref_span = 0;
    for (uint32_t k = 0; k < n_cig; k++) {
      uint32_t c = rd32(cig + 4 * k), op = c & 15, ln = c >> 4;
      if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) ref_span += (int32_t)ln;
    }
    if (pos + (ref_span > 0 ? ref_span : 1) <= start) continue;
    if (mapq == 0) continue;
    const uint8_t* tag = cig + 4 * (size_t)n_cig + ((size_t)l_seq + 1) / 2 + (size_t)l_seq;
    const uint8_t* rec_end = r + bs;
    int tp_primary = 0;
    while (tag + 3 <= rec_end) {
      char ty = (char)tag[2];
      const uint8_t* v = tag + 3;
      const size_t left = (size_t)(rec_end - v);
      size_t adv;
      if (ty == 'Z' || ty == 'H') {
        const void* z = memchr(v, 0, left);
        if (!z) { rc = fail(b, REC_ERR[E_TAG_UNTERM], (const char*)(r + 32), (long)ty); break; }
        adv = (size_t)((const uint8_t*)z - v) + 1;
      }
      else if (ty == 'A' || ty == 'c' || ty == 'C') { adv = 1; if (left >= 1 && tag[0] == 't' && tag[1] == 'p' && ty == 'A') tp_primary = (v[0] == 'P'); }
      else if (ty == 's' || ty == 'S') adv = 2;
      else if (ty == 'i' || ty == 'I' || ty == 'f') adv = 4;
      else if (ty == 'B') {
        if (left < 5) { rc = fail(b, REC_ERR[E_TAG_B], (const char*)(r + 32), (long)left); break; }
        const size_t esz = b_elem_size((char)v[0]);
        if (!esz) { rc = fail(b, REC_ERR[E_TAG_B], (const char*)(r + 32), (long)v[0]); break; }
        adv = 5 + (size_t)rd32(v + 1) * esz;
      }
      else { rc = fail(b, REC_ERR[E_TAG_TYPE], (const char*)(r + 32), ty); break; }
      if (adv > left) { rc = fail(b, REC_ERR[E_TAG_PAST], (const char*)(r + 32), (long)adv); break; }
      tag = v + adv;
    }
    if (rc) break;
    if (!tp_primary) continue;
    if (l_seq <= 0) { rc = fail(b, "%s has no SEQ: len(read.query_sequence) raises TypeError in the reference (%ld)", (const char*)(r + 32), 0); break; }
    if (out && n < cap) out[n] = l_seq;
    n++;
  }
  free(s.buf);
  *n_out = n;
  if (rc) return rc;
  if (n > cap) return HM_ERR_CAPACITY;
  return HM_OK;
}

/* ------------------------------------------------------------------ writer (tests, tools, bench) */
/* A packed batch back to a coordinate-sorted BAM + BAI: cs:Z short form (or MD:Z, see HM_BAM_TAGS_*), tp:A:P, query
 * names "read<id>", deleted bases written as "n" ("N" in MD; they are not stored).  Mirrors bamio.write_batch_bam;
 * exists so that the benchmark can put a contig-sized BAM on disk in seconds.  Not on the calling path. */
typedef struct { uint8_t* p; size_t n, cap; } wbuf_t;
static int wb_need(wbuf_t* w, size_t add) {
  if (w->n + add <= w->cap) return 0;
  size_t nc = w->cap ? w->cap : (1u << 20);
  while (nc < w->n + add) nc += nc / 2;
  uint8_t* np_ = (uint8_t*)realloc(w->p, nc);
  if (!np_) return -1;
  w->p = np_; w->cap = nc;
  return 0;
}
static void wb_u32(wbuf_t* w, uint32_t v) { w->p[w->n++] = (uint8_t)v; w->p[w->n++] = (uint8_t)(v >> 8); w->p[w->n++] = (uint8_t)(v >> 16); w->p[w->n++] = (uint8_t)(v >> 24); }
/* the smallest bin of the (min_shift, depth) scheme that holds [beg, end) (htslib's hts_reg2bin) */
static uint32_t reg2bin(int64_t beg, int64_t end, int min_shift, int depth) {
  --end;
  for (int l = depth, sh = min_shift; l > 0; l--, sh += 3)
    if (beg >> sh == end >> sh) return bin_first(l) + (uint32_t)(beg >> sh);
  return 0;
}
#define WBLK 0xff00u
typedef struct {
  const uint8_t* src; size_t n_src;
  uint8_t* dst;        /* n_blocks * 65536 */
  uint32_t* csize;
  size_t n_blocks, next;
  int level, error;
  pthread_mutex_t mu;
} deflate_job_t;
static void* deflate_worker(void* arg) {
  deflate_job_t* j = (deflate_job_t*)arg;
  for (;;) {
    pthread_mutex_lock(&j->mu);
    size_t i0 = j->next; j->next += 8;
    pthread_mutex_unlock(&j->mu);
    if (i0 >= j->n_blocks) break;
    for (size_t i = i0; i < i0 + 8 && i < j->n_blocks; i++) {
      const size_t off = i * WBLK, len = j->n_src - off < WBLK ? j->n_src - off : WBLK;
      uint8_t* o = j->dst + i * 65536;
      z_stream zs; memset(&zs, 0, sizeof(zs));
      if (deflateInit2(&zs, j->level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) { j->error = 1; return NULL; }
      zs.next_in = (Bytef*)(j->src + off); zs.avail_in = (uInt)len;
      zs.next_out = o + 18; zs.avail_out = 65536 - 18 - 8;
      if (deflate(&zs, Z_FINISH) != Z_STREAM_END) { deflateEnd(&zs); j->error = 1; return NULL; }
      const uint32_t clen = (uint32_t)zs.total_out, bsize = clen + 25;
      deflateEnd(&zs);
      static const uint8_t head[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
      memcpy(o, head, 16); o[16] = (uint8_t)bsize; o[17] = (uint8_t)(bsize >> 8);
      const uint32_t crc = block_crc(j->src + off, len);
      uint8_t* t = o + 18 + clen;
      t[0] = (uint8_t)crc; t[1] = (uint8_t)(crc >> 8); t[2] = (uint8_t)(crc >> 16); t[3] = (uint8_t)(crc >> 24);
      t[4] = (uint8_t)len; t[5] = (uint8_t)(len >> 8); t[6] = (uint8_t)(len >> 16); t[7] = (uint8_t)(len >> 24);
      j->csize[i] = bsize + 1;
    }
  }
  return NULL;
}

int hm_bam_write_batch(const char* path, const char* chrom, int32_t contig_len, const char* sample, const hm_read_batch* b,
                       int level, int threads) {
  return hm_bam_write_batch_tags(path, chrom, contig_len, sample, b, level, threads, HM_BAM_TAGS_CS);
}

int hm_bam_write_batch_tags(const char* path, const char* chrom, int32_t contig_len, const char* sample, const hm_read_batch* b,
                            int level, int threads, int tags) {
  return hm_bam_write_batch_index(path, chrom, contig_len, sample, b, level, threads, tags, 0, 0);
}

/* BGZF blocks of 0xff00 bytes of src, deflated on `threads` threads, then the end-of-file block, to f; coff (NULL: not
 * wanted) receives the file offset of every block, n_blocks + 1 entries */
static int bgzf_write(FILE* f, const uint8_t* src, size_t n, int level, int threads, uint64_t** coff_out) {
  deflate_job_t job; memset(&job, 0, sizeof(job));
  job.src = src; job.n_src = n; job.n_blocks = (n + WBLK - 1) / WBLK; job.level = level < 0 ? 1 : level;
  job.dst = (uint8_t*)malloc(job.n_blocks * 65536 + 1); job.csize = (uint32_t*)calloc(job.n_blocks + 1, 4);
  uint64_t* coff = (uint64_t*)malloc((job.n_blocks + 2) * sizeof(uint64_t));
  int rc = HM_OK;
  if (!job.dst || !job.csize || !coff) rc = HM_ERR_ARG;
  else {
    pthread_mutex_init(&job.mu, NULL);
    int nt = threads < 1 ? 1 : (threads > 64 ? 64 : threads);
    pthread_t th[64];
    for (int t = 1; t < nt; t++) pthread_create(&th[t], NULL, deflate_worker, &job);
    deflate_worker(&job);
    for (int t = 1; t < nt; t++) pthread_join(th[t], NULL);
    pthread_mutex_destroy(&job.mu);
    if (job.error) rc = HM_ERR_ARG;
    coff[0] = 0;
    for (size_t i = 0; i < job.n_blocks && !rc; i++) {
      if (fwrite(job.dst + i * 65536, 1, job.csize[i], f) != job.csize[i]) rc = HM_ERR_ARG;
      coff[i + 1] = coff[i] + job.csize[i];
    }
    static const uint8_t BGZF_EOF[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 0x42, 0x43, 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    if (!rc && fwrite(BGZF_EOF, 1, 28, f) != 28) rc = HM_ERR_ARG;
  }
  free(job.dst); free(job.csize);
  if (rc || !coff_out) free(coff);
  else *coff_out = coff;
  return rc;
}

typedef struct { uint32_t bin; uint64_t beg, end; size_t i; } bchunk_t;
static int cmp_chunk(const void* x, const void* y) {
  const bchunk_t *a = (const bchunk_t*)x, *c = (const bchunk_t*)y;
  return a->bin != c->bin ? (a->bin < c->bin ? -1 : 1) : (a->i < c->i ? -1 : a->i > c->i);
}

int hm_bam_write_batch_index(const char* path, const char* chrom, int32_t contig_len, const char* sample, const hm_read_batch* b,
                             int level, int threads, int tags, int min_shift, int depth) {
  if (!path || !chrom || !b || tags < HM_BAM_TAGS_CS || tags > HM_BAM_TAGS_M) return HM_ERR_ARG;
  const int csi = min_shift != 0;
  if (!csi && (int64_t)contig_len > ((int64_t)1 << 29)) return HM_ERR_ARG; /* past what a BAI can bin */
  if (csi) {
    if (depth <= 0) /* htslib's choice: the smallest depth whose span holds the contig plus 256 */
      for (depth = 0; ((int64_t)1 << (min_shift + 3 * depth)) < (int64_t)contig_len + 256; depth++) {}
    if (min_shift < 1 || depth > 10 || min_shift + 3 * depth > 62 || ((int64_t)1 << (min_shift + 3 * depth)) < (int64_t)contig_len) return HM_ERR_ARG;
  } else {
    min_shift = 14; depth = 5;
  }
  const int use_md = tags != HM_BAM_TAGS_CS;                             /* the walk below writes MD (unused without a tag) */
  const int no_tag = tags == HM_BAM_TAGS_EQX || tags == HM_BAM_TAGS_M;  /* no alignment tag: CIGAR + reference decodes it */
  const int m_cigar = tags == HM_BAM_TAGS_MD || tags == HM_BAM_TAGS_M;
  const uint32_t m_op = m_cigar ? 0 : 7, x_op = m_cigar ? 0 : 8;
  (void)hm_crc32_available(); /* probed before the deflate threads exist */
  wbuf_t w; memset(&w, 0, sizeof(w));
  char text[1024];
  int ltext = snprintf(text, sizeof(text), "@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:%s\tLN:%d\n@RG\tID:rg\tSM:%s\n", chrom, contig_len, sample ? sample : "synth");
  const size_t lname = strlen(chrom) + 1;
  if (wb_need(&w, 64 + (size_t)ltext + lname)) return HM_ERR_ARG;
  memcpy(w.p, "BAM\1", 4); w.n = 4; wb_u32(&w, (uint32_t)ltext); memcpy(w.p + w.n, text, (size_t)ltext); w.n += (size_t)ltext;
  wb_u32(&w, 1); wb_u32(&w, (uint32_t)lname); memcpy(w.p + w.n, chrom, lname); w.n += lname; wb_u32(&w, (uint32_t)contig_len);
  const size_t n = (size_t)b->n_reads;
  uint64_t* rec_off = (uint64_t*)malloc((n + 1) * sizeof(uint64_t));
  int32_t* rec_end = (int32_t*)malloc((n + 1) * sizeof(int32_t));
  char* cs = NULL; size_t cs_cap = 0;
  uint32_t* cig = NULL; size_t cig_cap = 0;
  int rc = HM_OK;
  static const char DEC[4] = {'a', 't', 'g', 'c'};
  static const uint8_t NIB[4] = {1, 8, 4, 2}; /* A T G C */
  for (size_t r = 0; r < n && !rc; r++) {
    const int32_t ql = b->qlen[r], qstart = b->qstart[r];
    const uint32_t nops = b->n_ops[r];
    const uint32_t* ops = b->ops + b->op_off[r];
    const uint8_t* seq = b->seq + b->seq_off[r];
    size_t need_cs = 16;
    for (uint32_t k = 0; k < nops; k++) { const uint32_t kind = ops[k] & 3u, v = ops[k] >> 2; need_cs += (kind == HM_OP_MATCH) ? 12 : (kind == HM_OP_SUB) ? 14 : (size_t)v + 14; }
    if (need_cs > cs_cap) { cs_cap = need_cs * 2; cs = (char*)realloc(cs, cs_cap); }
    if ((size_t)nops + 4 > cig_cap) { cig_cap = ((size_t)nops + 4) * 2; cig = (uint32_t*)realloc(cig, cig_cap * 4); }
    if (!cs || !cig) { rc = HM_ERR_ARG; break; }
    size_t lc = 0, ncig = 0;
    int32_t q = qstart, rspan = 0;
    uint32_t md_run = 0; /* MD: matched bases since the last event */
#define CIG(op, len) do { if (ncig && (cig[ncig - 1] & 15u) == (uint32_t)(op)) cig[ncig - 1] += (uint32_t)(len) << 4; else cig[ncig++] = ((uint32_t)(len) << 4) | (uint32_t)(op); } while (0)
    if (qstart) CIG(4, qstart);
    for (uint32_t k = 0; k < nops; k++) {
      const uint32_t kind = ops[k] & 3u, v = ops[k] >> 2;
      if (use_md) {
        if (kind == HM_OP_MATCH) { md_run += v; CIG(m_op, v); q += (int32_t)v; rspan += (int32_t)v; }
        else if (kind == HM_OP_SUB) { lc += (size_t)sprintf(cs + lc, "%u%c", md_run, (v & 7u) < 4 ? "ATGC"[v & 7u] : 'N'); md_run = 0; CIG(x_op, 1); q += 1; rspan += 1; }
        else if (kind == HM_OP_INS) { CIG(1, v); q += (int32_t)v; }
        else { lc += (size_t)sprintf(cs + lc, "%u^", md_run); md_run = 0; for (uint32_t i = 0; i < v; i++) cs[lc++] = 'N'; CIG(2, v); rspan += (int32_t)v; }
      }
      else if (kind == HM_OP_MATCH) { lc += (size_t)sprintf(cs + lc, ":%u", v); CIG(7, v); q += (int32_t)v; rspan += (int32_t)v; }
      else if (kind == HM_OP_SUB) { cs[lc++] = '*'; cs[lc++] = (v & 7u) < 4 ? DEC[v & 7u] : 'n'; cs[lc++] = DEC[(v >> 3) & 3u]; CIG(8, 1); q += 1; rspan += 1; }
      else if (kind == HM_OP_INS) { cs[lc++] = '+'; for (uint32_t i = 0; i < v; i++) { const int32_t qq = q + (int32_t)i; cs[lc++] = DEC[(seq[qq >> 2] >> (2 * (qq & 3))) & 3]; } CIG(1, v); q += (int32_t)v; }
      else { cs[lc++] = '-'; for (uint32_t i = 0; i < v; i++) cs[lc++] = 'n'; CIG(2, v); rspan += (int32_t)v; }
    }
    if (use_md) lc += (size_t)sprintf(cs + lc, "%u", md_run);
    if (ql - q > 0) CIG(4, ql - q);
#undef CIG
    cs[lc] = 0;
    char qname[32];
    const int lq = snprintf(qname, sizeof(qname), "read%u", b->qname_id[r]) + 1;
    const int32_t pos = b->tstart[r], endp = pos + (rspan > 0 ? rspan : 1);
    const size_t body = 32 + (size_t)lq + 4 * ncig + ((size_t)ql + 1) / 2 + (size_t)ql + (no_tag ? 0 : 3 + lc + 1) + 4;
    if (wb_need(&w, body + 8)) { rc = HM_ERR_ARG; break; }
    rec_off[r] = w.n; rec_end[r] = endp;
    wb_u32(&w, (uint32_t)body);
    wb_u32(&w, 0); wb_u32(&w, (uint32_t)pos);
    w.p[w.n++] = (uint8_t)lq; w.p[w.n++] = b->mapq[r];
    /* the BAI bin, which no decoder here reads: past 2^29 no BAI bin exists, and 4680 there cannot be right */
    const uint32_t bin = endp - 1 < (1 << 29) ? reg2bin(pos, endp, 14, 5) : 4680;
    w.p[w.n++] = (uint8_t)bin; w.p[w.n++] = (uint8_t)(bin >> 8);
    w.p[w.n++] = (uint8_t)ncig; w.p[w.n++] = (uint8_t)(ncig >> 8);
    const uint32_t flag = (b->flags[r] & HM_READ_SECONDARY) ? 0x100u : 0u;
    w.p[w.n++] = (uint8_t)flag; w.p[w.n++] = (uint8_t)(flag >> 8);
    wb_u32(&w, (uint32_t)ql); wb_u32(&w, 0xffffffffu); wb_u32(&w, 0xffffffffu); wb_u32(&w, 0);
    memcpy(w.p + w.n, qname, (size_t)lq); w.n += (size_t)lq;
    for (size_t k = 0; k < ncig; k++) wb_u32(&w, cig[k]);
    for (int32_t i = 0; i < ql; i += 2) {
      const uint8_t hi = NIB[(seq[i >> 2] >> (2 * (i & 3))) & 3];
      const uint8_t lo = (i + 1 < ql) ? NIB[(seq[(i + 1) >> 2] >> (2 * ((i + 1) & 3))) & 3] : 0;
      w.p[w.n++] = (uint8_t)((hi << 4) | lo);
    }
    memcpy(w.p + w.n, b->bq + b->bq_off[r], (size_t)ql); w.n += (size_t)ql;
    if (!no_tag) { w.p[w.n++] = use_md ? 'M' : 'c'; w.p[w.n++] = use_md ? 'D' : 's'; w.p[w.n++] = 'Z'; memcpy(w.p + w.n, cs, lc + 1); w.n += lc + 1; }
    w.p[w.n++] = 't'; w.p[w.n++] = 'p'; w.p[w.n++] = 'A'; w.p[w.n++] = 'P';
  }
  free(cs); free(cig);
  if (rc) { free(w.p); free(rec_off); free(rec_end); return rc; }
  rec_off[n] = w.n;
  FILE* f = fopen(path, "wb");
  uint64_t* coff = NULL;
  rc = f ? bgzf_write(f, w.p, w.n, level, threads, &coff) : HM_ERR_ARG;
  if (f && fclose(f)) rc = HM_ERR_ARG;
  /* the index: bins (adjacent records of one bin merged into one chunk) + linear index of 2^min_shift windows.  A BAI
   * keeps the linear index; a CSI keeps, per bin, the linear-index entry of its first window (its loffset, as htslib's
   * update_loff sets it) and comes BGZF-compressed. */
  bchunk_t* ch = NULL;
  uint64_t* lin = NULL;
  wbuf_t x; memset(&x, 0, sizeof(x));
  if (!rc) {
#define VOFF(o) ((coff[(o) / WBLK] << 16) | (uint64_t)((o) % WBLK))
    int64_t n_lin = 0;
    for (size_t r = 0; r < n; r++) if (((int64_t)rec_end[r] - 1) >> min_shift >= n_lin) n_lin = (((int64_t)rec_end[r] - 1) >> min_shift) + 1;
    if (!csi && contig_len > 0) n_lin = (((int64_t)contig_len - 1) >> 14) + 1;
    lin = (uint64_t*)calloc((size_t)n_lin + 1, 8);
    ch = (bchunk_t*)malloc((n + 1) * sizeof(bchunk_t));
    if (!lin || !ch) rc = HM_ERR_ARG;
    size_t nch = 0;
    for (size_t r = 0; r < n && !rc; r++) {
      const int64_t pos = b->tstart[r], endp = rec_end[r];
      const uint64_t v0 = VOFF(rec_off[r]), v1 = VOFF(rec_off[r + 1]);
      const uint32_t bin = reg2bin(pos, endp, min_shift, depth);
      if (nch && ch[nch - 1].bin == bin && ch[nch - 1].end == v0) ch[nch - 1].end = v1;
      else { ch[nch].bin = bin; ch[nch].beg = v0; ch[nch].end = v1; ch[nch].i = nch; nch++; }
      for (int64_t wv = pos >> min_shift; wv <= ((endp - 1) >> min_shift) && wv < n_lin; wv++) if (!lin[wv]) lin[wv] = v0;
    }
    if (!rc) {
      /* windows no record overlaps: a CSI (htslib) takes the contig's first record before the first one that has an
       * entry and the entry to the left after it; the BAI keeps 0 before the first entry */
      uint64_t last = csi && n ? VOFF(rec_off[0]) : 0;
      for (int64_t k = 0; k < n_lin; k++) { if (lin[k]) last = lin[k]; else lin[k] = last; }
      qsort(ch, nch, sizeof(bchunk_t), cmp_chunk);
      uint32_t n_bins = 0;
      for (size_t i = 0; i < nch; i++) if (i == 0 || ch[i].bin != ch[i - 1].bin) n_bins++;
      if (wb_need(&x, 128 + nch * 28 + (size_t)n_bins * 8 + (size_t)n_lin * 8)) rc = HM_ERR_ARG;
    }
    if (!rc) {
      memcpy(x.p, csi ? "CSI\1" : "BAI\1", 4); x.n = 4;
      if (csi) { wb_u32(&x, (uint32_t)min_shift); wb_u32(&x, (uint32_t)depth); wb_u32(&x, 0); }
      wb_u32(&x, 1);
      uint32_t n_bins = 0;
      for (size_t i = 0; i < nch; i++) if (i == 0 || ch[i].bin != ch[i - 1].bin) n_bins++;
      wb_u32(&x, n_bins + (csi && nch ? 1 : 0));
      for (size_t i = 0; i < nch;) {
        size_t j = i;
        while (j < nch && ch[j].bin == ch[i].bin) j++;
        wb_u32(&x, ch[i].bin);
        if (csi) {
          const int64_t bot = bin_start(ch[i].bin, min_shift, depth) >> min_shift;
          const uint64_t loff = bot < n_lin ? lin[bot] : 0;
          wb_u32(&x, (uint32_t)loff); wb_u32(&x, (uint32_t)(loff >> 32));
        }
        wb_u32(&x, (uint32_t)(j - i));
        for (size_t k = i; k < j; k++) {
          const uint64_t a = ch[k].beg, e = ch[k].end;
          wb_u32(&x, (uint32_t)a); wb_u32(&x, (uint32_t)(a >> 32)); wb_u32(&x, (uint32_t)e); wb_u32(&x, (uint32_t)(e >> 32));
        }
        i = j;
      }
      if (csi) {
        if (nch) { /* the pseudo-bin: the contig's first and last offsets, then mapped and unmapped record counts */
          const uint64_t pv[4] = {VOFF(rec_off[0]), VOFF(rec_off[n]), (uint64_t)n, 0};
          wb_u32(&x, pseudo_bin(depth)); wb_u32(&x, 0); wb_u32(&x, 0); wb_u32(&x, 2);
          for (int k = 0; k < 4; k++) { wb_u32(&x, (uint32_t)pv[k]); wb_u32(&x, (uint32_t)(pv[k] >> 32)); }
        }
      } else {
        wb_u32(&x, (uint32_t)n_lin);
        for (int64_t k = 0; k < n_lin; k++) { wb_u32(&x, (uint32_t)lin[k]); wb_u32(&x, (uint32_t)(lin[k] >> 32)); }
      }
      wb_u32(&x, 0); wb_u32(&x, 0); /* n_no_coor */
#undef VOFF
      char* ip = path_with(path, strlen(path), csi ? ".csi" : ".bai");
      FILE* g = ip ? fopen(ip, "wb") : NULL;
      free(ip);
      if (!g) rc = HM_ERR_ARG;
      else {
        if (csi) rc = bgzf_write(g, x.p, x.n, level, 1, NULL);
        else if (fwrite(x.p, 1, x.n, g) != x.n) rc = HM_ERR_ARG;
        if (fclose(g)) rc = HM_ERR_ARG;
      }
    }
  }
  free(lin); free(ch); free(x.p);
  free(w.p); free(rec_off); free(rec_end); free(coff);
  return rc;
}

/* ------------------------------------------------------------------ compact quality stream */
/* hm_bq_compact of a packed batch (include/himut_b200.h): bitmap of the modal quality + the exceptions.
 * mask (bq_bytes / 8 bytes) and exc_off (n_reads + 1) are caller allocated; exc is malloc'ed here and handed
 * over in *exc_out (free with hm_bq_compact_free).  The modal value is the most frequent quality of the batch. */
typedef struct {
  const hm_read_batch* b;
  uint8_t* mask; uint8_t* exc; uint64_t* exc_off;
  uint8_t modal;
  size_t next;
  int pass;
  pthread_mutex_t mu;
} bqc_job_t;
static void* bqc_worker(void* arg) {
  bqc_job_t* j = (bqc_job_t*)arg;
  const hm_read_batch* b = j->b;
  for (;;) {
    pthread_mutex_lock(&j->mu);
    size_t r0 = j->next; j->next += 256;
    pthread_mutex_unlock(&j->mu);
    if (r0 >= b->n_reads) break;
    for (size_t r = r0; r < r0 + 256 && r < b->n_reads; r++) {
      const uint8_t* q = b->bq + b->bq_off[r];
      const int32_t n = b->qlen[r];
      if (j->pass == 0) {
        uint64_t c = 0;
        for (int32_t i = 0; i < n; i++) c += (q[i] != j->modal);
        j->exc_off[r + 1] = c;
      } else {
        uint8_t* m = j->mask + (b->bq_off[r] >> 3);
        uint8_t* e = j->exc + j->exc_off[r];
        const size_t mb = (((size_t)n + 15) & ~(size_t)15) >> 3;
        memset(m, 0, mb);
        for (int32_t i = 0; i < n; i++) {
          if (q[i] == j->modal) m[i >> 3] |= (uint8_t)(1u << (i & 7));
          else *e++ = q[i];
        }
      }
    }
  }
  return NULL;
}
int hm_bq_compact_build(const hm_read_batch* b, int threads, uint8_t* mask, uint64_t* exc_off, uint8_t** exc_out,
                        uint64_t* exc_bytes, uint8_t* modal_out) {
  if (!b || !b->bq || !mask || !exc_off || !exc_out || !exc_bytes || !modal_out) return HM_ERR_ARG;
  uint64_t hist[256];
  memset(hist, 0, sizeof(hist));
  const uint64_t step = b->bq_bytes > (1u << 24) ? b->bq_bytes >> 22 : 1; /* a sample is enough to find the mode */
  for (uint64_t i = 0; i < b->bq_bytes; i += step) hist[b->bq[i]]++;
  int modal = 1;
  for (int v = 1; v < 256; v++) if (hist[v] > hist[modal]) modal = v;
  bqc_job_t job; memset(&job, 0, sizeof(job));
  job.b = b; job.mask = mask; job.exc_off = exc_off; job.modal = (uint8_t)modal;
  pthread_mutex_init(&job.mu, NULL);
  const int nt = threads < 1 ? 1 : (threads > 64 ? 64 : threads);
  pthread_t th[64];
  memset(mask, 0, (size_t)(b->bq_bytes >> 3));
  exc_off[0] = 0;
  for (int pass = 0; pass < 2; pass++) {
    job.pass = pass; job.next = 0;
    for (int t = 1; t < nt; t++) pthread_create(&th[t], NULL, bqc_worker, &job);
    bqc_worker(&job);
    for (int t = 1; t < nt; t++) pthread_join(th[t], NULL);
    if (pass == 0) {
      for (uint64_t r = 0; r < b->n_reads; r++) exc_off[r + 1] += exc_off[r];
      const uint64_t tot = exc_off[b->n_reads];
      job.exc = (uint8_t*)calloc(((size_t)tot + 31) & ~(size_t)15, 1);
      if (!job.exc) { pthread_mutex_destroy(&job.mu); return HM_ERR_ARG; }
      *exc_bytes = tot;
    }
  }
  pthread_mutex_destroy(&job.mu);
  *exc_out = job.exc; *modal_out = (uint8_t)modal;
  return HM_OK;
}
void hm_bq_compact_free(uint8_t* exc) { free(exc); }

/* test hook: the raw DEFLATE decoder of inflate_fast.h on one stream (0 = ok) */
int hm_inflate_raw_test(const uint8_t* in, size_t in_len, uint8_t* out, size_t out_len) { return hm_inflate_raw(in, in_len, out, out_len); }
int hm_inflate_raw2_test(const uint8_t* in0, size_t in_len0, uint8_t* out0, size_t out_len0, const uint8_t* in1, size_t in_len1, uint8_t* out1,
                         size_t out_len1) {
  int rc[2];
  hm_inflate_raw2(in0, in_len0, out0, out_len0, in1, in_len1, out1, out_len1, rc);
  return (rc[0] ? 1 : 0) | (rc[1] ? 2 : 0);
}

