/*
 * himut_io.h — C ABI of the native BAM region decoder (host side, no CUDA):
 * himut_b200/csrc/bamdec.c -> himut_b200/libhimut_io.so.
 *
 * SURVEY.md §8(f) row 1.  It replaces, for the GPU workers, what the reference does per record
 * through pysam / htslib and Python:
 *     alignments.fetch(chrom, start, end)          reference src/himut/caller.py:267,299
 *                                                  src/himut/normcounts.py:259,292
 *     bamlib.BAM.__init__ (9 attribute pulls)      reference src/himut/bamlib.py:15-32
 *     cslib.cs2lst / cs2tuple (regex over cs:Z)    reference src/himut/cslib.py:7-44
 * and hands back the packed structure-of-arrays batch of himut_b200.h directly, so no Python
 * object is created per record.  BGZF blocks are inflated by a pthread pool (zlib).
 *
 * Conventions: every function returns an int status (HM_OK == 0, codes of himut_b200.h);
 * hm_bam_error() gives the message.  A handle is single-threaded.  The arrays of a decoded
 * batch are owned by the handle and stay valid until the next hm_bam_read_batch / close.
 */
#ifndef HIMUT_IO_H
#define HIMUT_IO_H

#include "himut_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hm_bam hm_bam;

/* open <path> (and <path>.bai when it exists: without it every query scans from the first
 * record), read the header text and the @SQ table (bamlib.get_tname2tsize, bamlib.py:109-129) */
int hm_bam_open(const char* path, hm_bam** out);
void hm_bam_close(hm_bam* b);
const char* hm_bam_error(const hm_bam* b);

const char* hm_bam_header_text(const hm_bam* b); /* SAM header text, as str(alignments.header) */
int hm_bam_n_refs(const hm_bam* b);
const char* hm_bam_ref_name(const hm_bam* b, int i);
int hm_bam_ref_len(const hm_bam* b, int i);

/* the records of contig `rid` overlapping the 0-based half-open window [start, end), in file
 * order, each once (pysam fetch semantics, caller.py:299); secondary records (0x100) are
 * dropped as bamlib.BAM.__init__ drops them (bamlib.py:17), supplementary ones are kept.
 * Inputs the reference would crash on are rejected with HM_ERR_ARG and a message: no cs:Z tag,
 * missing qualities, a read base outside A/C/G/T under a cs match or as the substituted base, cs spans that
 * disagree with the CIGAR, records whose fields run past their block_size.  Hard-clipped records are decoded as pysam
 * presents them (SEQ holds no hard-clipped base; lead / trail count soft clips only).  `threads` = inflate threads. */
int hm_bam_read_batch(hm_bam* b, int rid, int32_t start, int32_t end, int threads, hm_read_batch* out);

/* HM_BAM_OPT_NO_SEQ = 1: batches come without the 2-bit base stream (seq = NULL, seq_off = NULL, seq_bytes = 0; see
 * hm_read_batch in himut_b200.h) — `call` and the phase edges do not need it; every check on the bases (A/C/G/T under
 * a cs match, long-form cs against SEQ) is still made.  Default 0. */
#define HM_BAM_OPT_NO_SEQ 1
/* HM_BAM_OPT_COMPACT_BQ = 1: the qualities of a batch come in the compact form of struct hm_bq_compact [himut_b200.h]: a bitmap
 * of the handle's modal quality + the other qualities in read order), written by the record-parse pass itself — no
 * one-byte-per-base stream is produced and no second pass is made; hm_read_batch.bq is NULL, bq_off / bq_bytes
 * describe the layout the device expands to.  hm_bam_last_compact fills the struct for hm_upload_batch_compact /
 * hm_call_batch_compact.  Default 0. */
#define HM_BAM_OPT_COMPACT_BQ 2
/* HM_BAM_OPT_BUFFER_SET = 0 | 1: which of the handle's two sets of output buffers the next hm_bam_read_batch fills.
 * The arrays of a batch stay valid until the next batch decoded into the same set, so a worker can upload one batch
 * while the next is decoded (query-name ids stay global: the name table is the handle's).  Default 0. */
#define HM_BAM_OPT_BUFFER_SET 3
int hm_bam_set_option(hm_bam* b, int option, int value);
/* the compact quality stream of the last batch decoded with HM_BAM_OPT_COMPACT_BQ (pointers into the handle's
 * buffers of the active set) */
int hm_bam_last_compact(hm_bam* b, hm_bq_compact* out);

/* BAM pre-pass of bamlib.get_thresholds (reference src/himut/bamlib.py:137-178): len(query_sequence) of
 * every record of contig `rid` that overlaps [start, end) with mapping_quality > 0 and tp:A:P, in fetch
 * order (secondary / supplementary records included: the reference does not test the flag there).  Only
 * record headers, CIGARs and tags are parsed.  HM_ERR_CAPACITY when cap is too small (*n_out = needed). */
int hm_bam_window_qlens(hm_bam* b, int rid, int32_t start, int32_t end, int threads, int32_t* out, size_t cap, size_t* n_out);

/* tests / tools / bench only: a packed batch back to a coordinate-sorted BAM + BAI (cs:Z short form, tp:A:P,
 * query names "read<qname_id>"), BGZF blocks deflated on `threads` threads at zlib `level` */
int hm_bam_write_batch(const char* path, const char* chrom, int32_t contig_len, const char* sample, const hm_read_batch* b,
                       int level, int threads);

/* compact quality stream of a packed batch (struct hm_bq_compact, himut_b200.h), for the host -> device copy: `mask` (bq_bytes / 8 bytes) and
 * `exc_off` (n_reads + 1 entries) are caller allocated, the exception bytes are allocated here (*exc_out, release
 * with hm_bq_compact_free); *modal_out is the batch's most frequent quality */
int hm_bq_compact_build(const hm_read_batch* b, int threads, uint8_t* mask, uint64_t* exc_off, uint8_t** exc_out,
                        uint64_t* exc_bytes, uint8_t* modal_out);
void hm_bq_compact_free(uint8_t* exc);

/* plan of the records hm_bam_read_batch would visit for [start, end) of contig `rid`, for the device decoder
 * (hm_decode_bam_begin of himut_b200.h): nothing is inflated.  The range starts at the BAI linear-index entry
 * hm_bam_read_batch seeks to and ends at the largest chunk end of the BAI bins that overlap the region; the entry
 * points are the linear-index entries of the windows the region covers.  Without a BAI: one entry point at the first
 * record and the range runs to the end of the file.  An empty contig gives n_entry = 0.  The arrays (and the
 * compressed range, when the file is not mapped) belong to the handle until its next plan. */
int hm_bam_region_plan(hm_bam* b, int rid, int32_t start, int32_t end, hm_bgzf_plan* out);
/* the ids of `n` NUL-terminated names (name i at blob + off[i]) in the handle's query-name table: the ids
 * hm_bam_read_batch gives the same names */
int hm_bam_intern_qnames(hm_bam* b, const char* blob, const uint64_t* off, size_t n, uint32_t* ids);

/* query names are interned per handle: qname_id of a batch indexes this table, ids are stable
 * across hm_bam_read_batch calls (m.num_ccs counts distinct names per contig, caller.py:318-320) */
uint32_t hm_bam_n_qnames(const hm_bam* b);
const char* hm_bam_qname(const hm_bam* b, uint32_t id);
/* the names of the ids whose flag byte is set (flags as hm_qname_seen returns them), each followed by '\n', in id order;
 * HM_ERR_CAPACITY with *need = bytes wanted when `out` is NULL or too small.  For workers that own a run of a contig's
 * chunks: the merge counts distinct names per contig across runs (genome.py) */
int hm_bam_qnames_blob(const hm_bam* b, const uint8_t* flags, size_t n_flags, char* out, size_t cap, size_t* need);

#ifdef __cplusplus
}
#endif
#endif
