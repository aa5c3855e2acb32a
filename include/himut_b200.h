/*
 * himut_b200.h — C ABI of the B200-native himut per-region calling hot path.
 *
 * The reference (sjin09/himut, pure Python) has no FFI of its own; the seam this
 * library sits behind is the pair of worker functions the reference hands to
 * multiprocessing.Pool.starmap:
 *     himut.caller.get_somatic_substitutions      (reference src/himut/caller.py:208-642)
 *     himut.normcounts.get_callable_tricounts     (reference src/himut/normcounts.py:206-420)
 * The Python mirrors of those two functions (himut_b200/caller.py, himut_b200/normcounts.py)
 * decode a contig's alignments into the packed structure-of-arrays batch below and call
 * the entry points declared here through ctypes.  Everything in this header is plain C:
 * pointers, sizes and PODs; no torch / CUDA types cross the boundary.
 *
 * Conventions
 *   - every function returns an int status (HM_OK == 0); hm_last_error() gives a message;
 *   - a context is single-threaded, one per (process, GPU); independent contexts may run
 *     concurrently;  nothing is initialised before hm_create (fork-safe: create the context
 *     inside the worker process);
 *   - all input buffers are caller-owned host memory (pinned memory makes the copies faster,
 *     it is not required); outputs are caller-allocated with a capacity, overflow returns
 *     HM_ERR_CAPACITY and writes the required size to *n_out;
 *   - allele / base codes follow the reference's util.base2idx (src/himut/util.py:14-20):
 *     A=0 T=1 G=2 C=3, insertion=4, deletion=5;  HM_BASE_N=4 only appears as the *reference*
 *     base of a substitution op.
 *
 * The same structs are consumed by the CPU oracle (oracle/himut_oracle.c), which is test
 * infrastructure only and is never linked into this library.
 */
#ifndef HIMUT_B200_H
#define HIMUT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HM_ABI_VERSION 1

/* ---- status codes ------------------------------------------------------------------ */
enum {
  HM_OK = 0,
  HM_ERR_ARG = 1,        /* bad argument / malformed batch                                  */
  HM_ERR_CUDA = 2,       /* CUDA runtime failure (message has the CUDA error string)        */
  HM_ERR_CAPACITY = 3,   /* output buffer too small; *n_out holds the size needed           */
  HM_ERR_BQ_ZERO = 4,    /* a base quality of 0 reached the genotype model: the reference
                            raises ValueError there (math.log10(0), gtlib.py:52-65)         */
  HM_ERR_NO_DEVICE = 5,  /* no usable CUDA device                                           */
  HM_ERR_STATE = 6       /* call order violated (e.g. params not set)                       */
};

/* ---- cs-tag op stream -------------------------------------------------------------- */
/* One u32 per cs token (reference cslib.cs2tuple, src/himut/cslib.py:13-44):
 *   bits 0..1  kind: 0 match (":n" / "=SEQ"), 1 substitution ("*xy"), 2 insertion ("+seq"),
 *                    3 deletion ("-seq")
 *   bits 2..31 value: run length for match / insertion / deletion;
 *                     for a substitution  ref_code | alt_code << 3   (codes above, N = 4)   */
#define HM_OP_MATCH 0u
#define HM_OP_SUB 1u
#define HM_OP_INS 2u
#define HM_OP_DEL 3u
#define HM_BASE_N 4u
#define HM_MAKE_OP(kind, value) ((uint32_t)(kind) | ((uint32_t)(value) << 2))
#define HM_MAKE_SUB(ref_code, alt_code) HM_MAKE_OP(HM_OP_SUB, (uint32_t)(ref_code) | ((uint32_t)(alt_code) << 3))

/* read flag bits (hm_read_batch.flags) */
#define HM_READ_SECONDARY 1u /* pysam is_secondary (0x100): skipped everywhere, bamlib.py:17 */

/* ---- packed structure-of-arrays read batch (one contig) --------------------------- */
/* Reads are in BAM file order (coordinate sorted: tstart non-decreasing).  Each read is
 * stored once; chunks address them by index range.  Replaces the per-record attribute
 * pulls of bamlib.BAM.__init__ (src/himut/bamlib.py:15-32).                                */
typedef struct hm_read_batch {
  uint64_t n_reads;
  const int32_t* tstart;    /* reference_start, 0-based                                     */
  const int32_t* tend;      /* reference_end, 0-based exclusive                             */
  const int32_t* qstart;    /* query_alignment_start (= leading soft clip)                  */
  const int32_t* qlen;      /* len(query_sequence), soft clips included                     */
  const uint8_t* mapq;
  const uint8_t* flags;     /* HM_READ_* bits                                               */
  const uint32_t* qname_id; /* equal ids <=> equal query names                              */
  const uint64_t* seq_off;  /* byte offset of the read's first base in `seq`, 16 B aligned  */
  const uint64_t* bq_off;   /* byte offset of the read's first quality in `bq`, 16 B aligned*/
  const uint64_t* op_off;   /* index of the read's first op in `ops`                        */
  const uint32_t* n_ops;
  const uint8_t* seq;       /* 2-bit bases, 4 per byte, base i at bits 2*(i&3) of byte i>>2 */
  uint64_t seq_bytes;       /* padded to a multiple of 16                                   */
                            /* seq may be NULL (seq_bytes 0, seq_off ignored): the batch then
                             * carries no base stream.  Substituted bases travel in the ops; the
                             * bases of match runs are, by the meaning of a cs match
                             * (cslib.py:22-29), the reference allele of the site that asks.
                             * hm_call_* and hm_phase_edges_* accept such a batch (a quarter of
                             * the upload less); hm_normcounts_chunks returns HM_ERR_STATE.   */
  const uint8_t* bq;        /* one byte per base                                            */
  uint64_t bq_bytes;        /* padded to a multiple of 16                                   */
  const uint32_t* ops;
  uint64_t n_ops_total;
} hm_read_batch;

/* Optional compact form of the quality stream for the host -> device copy.  CCS qualities are dominated by one
 * value (the Q93 cap), so `bq` (1 byte per base, 80 % of a batch) travels as a bitmap plus the exceptions and is
 * expanded on the device (k_bq_expand) into exactly the layout bq_off / bq_bytes describe.  Lossless.
 *   mask  one bit per byte of the expanded stream, padding included: bit (i & 7) of byte i >> 3 is set when byte i
 *         holds `modal`; bits of padding bytes are clear
 *   exc   the qualities whose bit is clear, read by read, in base order (padding excluded);
 *         read r's exceptions start at exc[exc_off[r]], exc_off has n_reads + 1 entries                          */
typedef struct hm_bq_compact {
  const uint8_t* mask;
  uint64_t mask_bytes;     /* bq_bytes / 8 */
  const uint8_t* exc;
  uint64_t exc_bytes;
  const uint64_t* exc_off;
  uint8_t modal;
  uint8_t reserved[7];
} hm_bq_compact;

/* One unit of work = one element of the reference's chunkloci_lst (util.chunkloci,
 * src/himut/util.py:119-132) or, in --phase mode, one phase-set span
 * (vcflib.load_phased_hetsnps, src/himut/vcflib.py:655-662).  `read_lo..read_hi` is the
 * smallest file-order index range that contains every record pysam's
 * fetch(chrom, start, end) would return; the library re-applies the overlap rule
 * tstart < end && tend > start inside the range.                                           */
/* A BAM region planned for the device decoder (hm_bam_region_plan of himut_io.h fills it, hm_decode_bam_begin reads
 * it): whole BGZF blocks of the file and the points of their inflated stream where a record is known to start.
 * Offsets into the inflated stream count from the first block of the range.  Valid until the next plan of the handle. */
typedef struct hm_bgzf_plan {
  const uint8_t* comp;        /* the compressed range (n_blocks whole BGZF blocks)                         */
  uint64_t comp_bytes;
  uint64_t n_blocks;
  const uint64_t* blk_coff;   /* n_blocks + 1: offset of each block in comp (last: comp_bytes)             */
  const uint32_t* blk_csize;  /* whole block size (BSIZE + 1)                                              */
  const uint32_t* blk_isize;  /* ISIZE of the footer                                                       */
  const uint64_t* blk_uoff;   /* n_blocks + 1: offset of the block's payload in the inflated stream        */
  const uint32_t* blk_crc;    /* CRC32 of the footer                                                       */
  const uint64_t* entry;      /* ascending inflated offsets of record starts (BAI linear index entries)    */
  uint64_t n_entry;           /* 0: nothing to decode                                                      */
  uint64_t walk_end;          /* records are walked up to this inflated offset                             */
  const char* path;           /* the BAM file, for messages                                                */
} hm_bgzf_plan;

typedef struct hm_chunk {
  int32_t start;
  int32_t end;
  uint32_t read_lo;
  uint32_t read_hi;
  int32_t phase_set; /* index into the phase-set table, -1 when not phasing                 */
  int32_t reserved;
} hm_chunk;

/* ---- parameters -------------------------------------------------------------------- */
/* The subset of the worker arguments the arithmetic uses (caller.py:208-241,
 * normcounts.py:206-238).  The three per-BQ tables hold the reference's own genotype
 * terms (gtlib.py:47-69) evaluated on the host for bq = 0..255:
 *   lut_hom[bq] = log10(1 - 10**(-bq/10)), lut_het[bq] = log10(0.5 - 10**(-bq/10)/2),
 *   lut_err[bq] = log10(10**(-(bq/3)/10));  entry 0 is never read (HM_ERR_BQ_ZERO).
 * log10_prior = log10 of gtlib.init's priors in the order homref, het, hetalt, homalt.     */
typedef struct hm_params {
  int32_t min_qv;
  int32_t min_mapq;
  int32_t qlen_lower_limit;
  int32_t qlen_upper_limit;
  int32_t min_gq;
  int32_t min_bq;
  int32_t max_mismatch_count;
  int32_t mismatch_window;
  int32_t min_ref_count;
  int32_t min_alt_count;
  int32_t min_hap_count;
  int32_t phase;
  int32_t non_human_sample;
  int32_t create_panel_of_normals;
  double min_sequence_identity;
  double min_trim;
  double md_threshold;
  double log10_prior[4];
  double lut_hom[256];
  double lut_het[256];
  double lut_err[256];
} hm_params;

/* ---- `himut call` outputs ----------------------------------------------------------- */
/* site status, in the order of the reference's cascade (caller.py:338-621) */
enum {
  HM_ST_PASS = 0,
  HM_ST_GERM_HET = 1,     /* candidate restates the germline genotype: counted, not emitted */
  HM_ST_GERM_HETALT = 2,
  HM_ST_GERM_HOMALT = 3,
  HM_ST_GERM_HOMREF = 4,  /* is_germ_gt true in the homref branch (alt == ref): no counter   */
  HM_ST_HET_SITE = 5,
  HM_ST_HETALT_SITE = 6,
  HM_ST_HOMALT_SITE = 7,
  HM_ST_INDEL_SITE = 8,
  HM_ST_LOW_GQ = 9,
  HM_ST_LOW_BQ = 10,
  HM_ST_PON = 11,
  HM_ST_COMSNP = 12,
  HM_ST_LOW_DEPTH = 13,
  HM_ST_HIGH_DEPTH = 14,
  HM_ST_UNPHASED = 15
};

/* hm_site_record.flags */
#define HM_SITE_PL_TIE 1u /* PL[best] == PL[second]: np.argsort's pick is platform dependent
                             in the reference (gtlib.py:113-119); we take the lowest
                             gt_lst index and flag the record                               */

/* One evaluated candidate (tpos, ref, alt) of one chunk.  Integers only: the Python side
 * derives alt_bq = bq_sum/count, vaf = count/depth and the strings, so formatting stays
 * in reference code (caller.py:349-621, vcflib.dump_sbs).                                   */
typedef struct hm_site_record {
  int32_t tpos;        /* 1-based                                                            */
  uint8_t ref;         /* base code                                                          */
  uint8_t alt;
  uint8_t status;      /* HM_ST_*                                                            */
  uint8_t flags;       /* HM_SITE_*                                                          */
  int32_t chunk;       /* index of the chunk that evaluated it                               */
  int32_t gq;          /* germ_gq (gtlib.get_germ_gq)                                        */
  uint8_t germ_gt[2];  /* germline genotype alleles after the ref-first flip (gtlib.py:133)  */
  uint8_t germ_state;  /* 0 homref 1 het 2 hetalt 3 homalt                                   */
  uint8_t pad0;
  int32_t counts[6];   /* rpos2allelecounts[tpos-1] (caller.py:44-72)                        */
  int32_t bq_sum[4];   /* sum of rpos2allele2bq_lst[tpos-1][allele]                          */
  int32_t hap_count[2];/* --phase: h0 / h1 counts among ref-allele reads (caller.py:556-570) */
  int32_t som_hap_mask;/* --phase: bit0 hap "0", bit1 hap "1" seen among alt-allele reads    */
  int32_t phase_set;   /* --phase: chunk_start of the phase set for PASS rows, else -1       */
} hm_site_record;

/* chrom2tsbs_log[chrom] (caller.py:625-641), same order */
#define HM_CALL_LOG_LEN 15
/* chrom2norm_log[chrom] (normcounts.py:404-419), same order */
#define HM_NORM_LOG_LEN 14
/* 32 pyrimidine-centred trinucleotides in mutlib.tri_lst order (src/himut/mutlib.py:17-50)
 * + one bin for contexts that contain N (tallied by the reference, never read back).       */
#define HM_TRI_BINS 33

/* ---- entry points -------------------------------------------------------------------- */
typedef struct hm_ctx hm_ctx;

int hm_abi_version(void);
/* visible CUDA devices (cudaGetDeviceCount; 0 without a driver or a device): pool workers place themselves with it */
int hm_device_count(void);
/* sizeof of the ABI structs as the library was compiled: 0 hm_read_batch, 1 hm_chunk,
 * 2 hm_params, 3 hm_site_record (bindings check their own layout against it) */
size_t hm_abi_sizeof(int which);

/* create / destroy a context bound to one CUDA device */
int hm_create(int cuda_device, hm_ctx** out);
void hm_destroy(hm_ctx* ctx);
const char* hm_last_error(const hm_ctx* ctx);

/* run the context's work on a caller-owned CUDA stream (a cudaStream_t passed as void*), so
 * the caller's own events bracket it; NULL goes back to the context's private stream */
int hm_set_stream(hm_ctx* ctx, void* cuda_stream);

/* page-lock / unlock caller memory (cudaHostRegister) so hm_upload_batch copies at PCIe speed */
int hm_host_register(hm_ctx* ctx, void* p, size_t bytes);
int hm_host_unregister(hm_ctx* ctx, void* p);

/* worker arguments (copied) */
int hm_set_params(hm_ctx* ctx, const hm_params* params);

/* common-SNP / panel-of-normals membership sets of the current contig, as sorted arrays of
 * keys  pos(1-based) << 4 | ref_code << 2 | alt_code   (replaces the Python sets built by
 * vcflib.load_common_snp / load_pon / load_bgz_*, src/himut/vcflib.py:356-459).            */
int hm_set_site_sets(hm_ctx* ctx, const uint64_t* common_sorted, size_t n_common,
                     const uint64_t* pon_sorted, size_t n_pon);

/* phased hetSNPs of the current contig (vcflib.load_phased_hetsnps): phase set s owns
 * entries set_off[s] .. set_off[s+1]; hpos is 1-based and ascending inside a set; hbit is
 * the h0 bit (0/1); set_id[s] is the set's chunk_start (the reference's phase_set key).
 * href / halt: base codes 0..3; 255 = an allele no read base can equal (an indel allele: the reference compares
 * the read's one-letter base with the allele string, haplib.py:46-58); href 16 + c = REF can never be equal but its
 * first base is c — what a batch without a base stream shows in a cs match run at that position.               */
int hm_set_phase_sets(hm_ctx* ctx, const int32_t* hpos, const uint8_t* href,
                      const uint8_t* halt, const uint8_t* hbit, size_t n_hetsnp,
                      const uint64_t* set_off, size_t n_sets);

/* upload a batch (H2D on the context's stream) and keep it resident until the next upload */
int hm_upload_batch(hm_ctx* ctx, const hm_read_batch* batch);

/* `himut call` over chunks of the resident batch (replaces the body of
 * caller.get_somatic_substitutions, caller.py:243-641).  Records come back in no particular
 * order; germline-restatement records are included (the host needs them for the counters).
 * log[15] follows chrom2tsbs_log.  n_tie, if not NULL, receives the number of flagged ties.*/
int hm_call_chunks(hm_ctx* ctx, const hm_chunk* chunks, size_t n_chunks,
                   hm_site_record* out, size_t cap, size_t* n_out,
                   int64_t log[HM_CALL_LOG_LEN]);

/* hm_call_chunks that returns as soon as the counters and *n_out are final: the copy of the records into `out` may
 * still be in flight (on a copy stream of the context) and overlaps whatever the caller enqueues next — a worker
 * that feeds a contig in several batches decodes / uploads / scans the next one meanwhile.  hm_records_wait blocks
 * until the records of every earlier call are complete.  At most two calls may be in flight: an `out` buffer must
 * not be reused before the second next call.  `out` must hold all records (HM_ERR_CAPACITY behaves as above, and
 * then synchronously).                                                                                          */
int hm_call_chunks_async(hm_ctx* ctx, const hm_chunk* chunks, size_t n_chunks,
                         hm_site_record* out, size_t cap, size_t* n_out,
                         int64_t log[HM_CALL_LOG_LEN]);
int hm_records_wait(hm_ctx* ctx);

/* hm_call_chunks_async in two halves, for a host that drives several contexts on one GPU (the chunk runs of a genome,
 * himut_b200/genome.py): submit enqueues the whole device path of the call on the context's stream and returns at once
 * (the fused path synchronises nowhere in between); collect waits for it and does the rest (counters, som_seen replay,
 * record copy, with hm_call_chunks_async's rules for `out`).  Submitting the calls of all contexts before collecting
 * the first keeps the device busy across them.  One call may be pending per context and nothing else may be asked
 * of the context until it is collected. */
int hm_call_chunks_submit(hm_ctx* ctx, const hm_chunk* chunks, size_t n_chunks);
int hm_call_chunks_collect(hm_ctx* ctx, hm_site_record* out, size_t cap, size_t* n_out, int64_t log[HM_CALL_LOG_LEN]);

/* options of a context.  HM_OPT_OMIT_RESTATEMENTS (default 0): records whose status is one of HM_ST_GERM_* — a
 * candidate that merely restates the germline genotype, which the reference counts and drops (caller.py:338-345) —
 * are not copied to the host; they still count in log[2..4].  A third of the record bytes at 30x.                */
#define HM_OPT_OMIT_RESTATEMENTS 1
/* HM_OPT_KERNEL_TIMING (default 1): CUDA events around the kernels of a call, read back by hm_last_timing /
 * hm_last_kernel_times.  0 saves the event records (a dozen driver calls per call); the figures are then not updated. */
#define HM_OPT_KERNEL_TIMING 2
int hm_set_option(hm_ctx* ctx, int option, int value);

/* after hm_call_chunks / hm_call_batch returned HM_ERR_CAPACITY: copy the records of that call
 * into a buffer of at least *n_out entries, without recomputing anything */
int hm_last_records(hm_ctx* ctx, hm_site_record* out, size_t cap, size_t* n_out);

/* convenience: upload + call in one step (the end-to-end path bench.py times) */
int hm_call_batch(hm_ctx* ctx, const hm_read_batch* batch, const hm_chunk* chunks,
                  size_t n_chunks, hm_site_record* out, size_t cap, size_t* n_out,
                  int64_t log[HM_CALL_LOG_LEN]);

/* hm_upload_batch / hm_call_batch with the quality stream in compact form (hm_bq_compact above): batch->bq is
 * ignored (may be NULL); batch->bq_off / bq_bytes still describe the expanded layout */
int hm_upload_batch_compact(hm_ctx* ctx, const hm_read_batch* batch, const hm_bq_compact* bq);
int hm_call_batch_compact(hm_ctx* ctx, const hm_read_batch* batch, const hm_bq_compact* bq, const hm_chunk* chunks,
                          size_t n_chunks, hm_site_record* out, size_t cap, size_t* n_out, int64_t log[HM_CALL_LOG_LEN]);

/* hm_upload_batch_compact in two halves: _begin returns as soon as the host -> device copies are enqueued (the buffers
 * of `batch` and `bq` must stay untouched until hm_upload_wait, the next hm_upload_* or hm_destroy of the context has
 * returned; calls enqueued meanwhile run behind the copies), hm_upload_wait returns when they are done.  A worker that
 * alternates two contexts between the decode groups of a contig (caller.py:268-299 is the loop this replaces) begins
 * the upload of group k + 1 on one context before it waits for group k's on the other and hands its buffers back to
 * the decoder. */
int hm_upload_batch_compact_begin(hm_ctx* ctx, const hm_read_batch* batch, const hm_bq_compact* bq);
int hm_upload_wait(hm_ctx* ctx);

/* keep a contig's reference sequence (the `seq` argument of get_callable_tricounts,
 * normcounts.py:208) resident on the device; hm_normcounts_chunks then accepts refseq = NULL */
int hm_set_reference(hm_ctx* ctx, const uint8_t* refseq, size_t ref_len);

/* callable-base half of `himut normcounts` over chunks of the resident batch (replaces the
 * body of normcounts.get_callable_tricounts, normcounts.py:240-419).  refseq is the contig
 * as upper/lower-case ASCII (positions outside A/T/G/C upper-case are skipped as in
 * normcounts.py:320).  n_alt_tie, if not NULL, receives the number of positions whose
 * max-count alt was tied (set-iteration order in the reference, normcounts.py:370-388).    */
int hm_normcounts_chunks(hm_ctx* ctx, const uint8_t* refseq, size_t ref_len,
                         const hm_chunk* chunks, size_t n_chunks,
                         int64_t ccs_tri[HM_TRI_BINS], int64_t ref_tri[HM_TRI_BINS],
                         int64_t log[HM_NORM_LOG_LEN], int64_t* n_alt_tie);

/* after hm_call_chunks / hm_normcounts_chunks: one byte per qname_id (0 .. max id of the batch),
 * 1 where a record with that id passed the read gates in a chunk that fetched it — the reads
 * m.num_ccs counts (caller.py:318-320).  Lets a host that feeds a contig in several batches
 * count distinct names across them.                                                          */
int hm_qname_seen(hm_ctx* ctx, uint8_t* out, size_t cap, size_t* n);

/* diagnostics: how many positions the last hm_normcounts_chunks evaluated with the exact ordered
 * fp64 genotype arithmetic; all the others were pure-reference positions whose verdict the integer
 * pass certified (DESIGN.md §4).  0 when the single-pass kernel ran.                            */
int hm_last_norm_exact_sites(hm_ctx* ctx, uint64_t* n);

/* ---- `himut phase`: hetSNP pair tables (replaces phaselib.get_edges, src/himut/phaselib.py:16-67) -------
 * hpos: ascending 1-based hetSNP positions of the contig (vcflib.load_hetsnps), href: their reference base codes
 * (4 = anything the read can never equal).  For every non-secondary read of the resident batch with
 * mapq >= min_mapq and reference_start >= min_tstart (so that a read shared by two decoded windows of a contig
 * is counted once) that covers at least two hetSNPs, every ordered pair a < b of them whose bases both have
 * BQ >= min_bq adds one to  counts[(a * band + (b - a - 1)) * 4 + k],  k = 0 cis1 (ref, ref), 1 cis2
 * (non-ref, non-ref), 2 trans1 (ref, non-ref), 3 trans2 (non-ref, ref); a, b index hpos.
 * begin zeroes the table on the device, add accumulates one resident batch (HM_ERR_CAPACITY and *need_band when a
 * read pairs hetSNPs further apart than the band: begin again with a wider one), end copies n_hetsnp * band * 4
 * counters out.                                                                                              */
int hm_phase_edges_begin(hm_ctx* ctx, const int32_t* hpos, const uint8_t* href, size_t n_hetsnp, uint32_t band);
int hm_phase_edges_add(hm_ctx* ctx, int32_t min_bq, int32_t min_mapq, int32_t min_tstart, uint32_t* need_band);
int hm_phase_edges_end(hm_ctx* ctx, uint32_t* counts, size_t cap_entries);

/* reference-genome trinucleotide counts of one contig, bins as above (replaces
 * reflib.get_chrom_tricount, src/himut/reflib.py:11-33: windows whose first base is "N" are skipped) */
int hm_ref_tricounts(hm_ctx* ctx, const uint8_t* refseq, size_t ref_len, int64_t tri[HM_TRI_BINS]);

/* per-read statistics of the resident batch, for parity tests of the expansion kernel
 * (cslib.cs2subindel / bamlib.get_blast_sequence_identity / BAM.get_qv):
 * bq_total = sum of all base qualities, n_match / n_sub / ins_len / del_len as in
 * bamlib.py:47-63, n_mismatch = len(ccs.mismatch_lst).  Any pointer may be NULL.           */
int hm_read_stats(hm_ctx* ctx, int64_t* bq_total, int32_t* n_match, int32_t* n_sub,
                  int32_t* ins_len, int32_t* del_len, int32_t* n_mismatch);

/* timing of the last hm_call_chunks / hm_normcounts_chunks on the context's stream (CUDA
 * events): total device milliseconds and the number of own kernels the call launched (fused `call` path: counted
 * launch by launch; elsewhere: the number of timed kernel groups).  names/ms give per-kernel
 * figures for up to `cap` kernels; returns how many were written in *n.                    */
/* Device BAM decoder: a region planned on the host (hm_bgzf_plan, hm_bam_region_plan of himut_io.h) becomes a
 * resident batch without being inflated on the host: the batch of `call` and the phase edges (no base stream), or with
 * HM_DECODE_SEQ the batch of normcounts (with the 2-bit base stream).  In two halves, so that a worker can decode the
 * next group on one context while the kernels of the current one run on another:
 *   hm_decode_bam_begin copies the compressed range up (cudaMemcpyAsync), inflates every BGZF block (CRC32 and
 *   ISIZE checked), walks the records from the entry points, selects and parses them with hm_bam_read_batch's rules
 *   (file order, same messages for rejected input: HM_ERR_ARG) and brings back the query names and the per-read
 *   coordinates; *n_reads = the batch's reads.  `end` is clamped to the contig by the caller.  It decodes without the
 *   base stream; hm_decode_bam_begin_opts takes option bits (HM_DECODE_SEQ; others: HM_ERR_ARG).
 *   hm_decode_bam_names: views of those host arrays (valid until the next begin): NUL-terminated names at
 *   names + name_off[i], tstart / tend per read.
 *   hm_decode_bam_end takes the query-name ids (interned by the BAM handle: hm_bam_intern_qnames) and makes the batch
 *   resident; afterwards every call behaves as after hm_upload_batch of hm_bam_read_batch's batch without seq, or
 *   with HM_DECODE_SEQ of its batch with seq (one quality byte per base either way). */
#define HM_DECODE_SEQ 1u /* hm_decode_bam_begin_opts: pack the 2-bit base stream too (seq / seq_off of hm_read_batch) */
int hm_decode_bam_begin(hm_ctx* ctx, const hm_bgzf_plan* plan, int rid, int32_t start, int32_t end, uint64_t* n_reads);
int hm_decode_bam_begin_opts(hm_ctx* ctx, const hm_bgzf_plan* plan, int rid, int32_t start, int32_t end, uint32_t opts,
                             uint64_t* n_reads);
int hm_decode_bam_names(hm_ctx* ctx, const char** names, const uint64_t** name_off, const int32_t** tstart,
                        const int32_t** tend, uint64_t* n_reads);
int hm_decode_bam_end(hm_ctx* ctx, const uint32_t* qname_id);

/* diagnostics (tests): the resident batch back into caller buffers (any may be NULL); *out gets n_reads, bq_bytes and
 * n_ops_total, which size them */
int hm_batch_read_back(hm_ctx* ctx, hm_read_batch* out, int32_t* tstart, int32_t* tend, int32_t* qstart, int32_t* qlen,
                       uint8_t* mapq, uint32_t* qname_id, uint64_t* bq_off, uint64_t* op_off, uint32_t* n_ops, uint8_t* bq,
                       uint32_t* ops);
/* diagnostics (tests): the resident base stream back into caller buffers (either may be NULL): n_reads offsets and
 * *seq_bytes bytes; *seq_bytes = 0 when the resident batch has none */
int hm_batch_read_back_seq(hm_ctx* ctx, uint64_t* seq_off, uint8_t* seq, uint64_t* seq_bytes);
/* tests: the device inflate of one raw DEFLATE stream (exactly out_len bytes, CRC32 crc); 0 ok, else an error code */
int hm_inflate_device_test(hm_ctx* ctx, const uint8_t* in, size_t in_len, uint8_t* out, size_t out_len, uint32_t crc);

int hm_last_timing(hm_ctx* ctx, float* total_ms, int* n_launches);
/* which device path the last hm_call_chunks took: 2 the fused one (no pass over the quality stream, no library
 * sort, one synchronisation), 1 the first version (chunk spans of 2^27 positions and more, or HIMUT_B200_CALL_V1 set),
 * 0 none yet.  Same records either way; for tests and bench.py.                                              */
int hm_last_call_path(hm_ctx* ctx);
int hm_last_kernel_times(hm_ctx* ctx, const char** names, float* ms, size_t cap, size_t* n);

#ifdef __cplusplus
}
#endif
#endif /* HIMUT_B200_H */
