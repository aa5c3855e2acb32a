// himut_b200.cu — context, device memory, launches and the C ABI of include/himut_b200.h.
//
// Host work kept here on purpose (it is sequential by definition in the reference):
//   - the som_seen carry between chunks of a contig (caller.py:243,347; bamlib.py:77):
//     the device evaluates every chunk independently, the host replays chunk order and
//     drops sites a previous chunk already claimed;
//   - the 15 / 14 log counters, summed from record statuses.
// Everything per base / per read / per site runs in the kernels of kernels.cuh and
// normcounts.cuh.  There is no CPU fallback: without a CUDA device hm_create fails.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_set>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>

#include "kernels.cuh"
#include "normcounts.cuh"
#include "normfast.cuh"
#include "callfused.cuh"
#include "normbits.cuh"
#include "bamgpu.cuh"

#define HM_BOUNDARY_CAP_DEFAULT 65536   // boundary records the device list holds (HIMUT_B200_BOUNDARY_CAP overrides: tests)
#define HM_BOUNDARY_FIRST 2048  // ... of which this many travel with the counters

namespace {

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// a host array in page-locked memory that grows like a vector: the library's own per-read tables are uploaded from it
// without a staging copy, so an upload that is not waited for (hm_upload_batch_compact_begin) never blocks the host
template <typename T>
struct PinVec {
  T* p = nullptr;
  size_t cap = 0, n = 0;
  bool resize(size_t m) { // false: out of page-locked memory
    if (m > cap) {
      if (p) cudaFreeHost(p);
      p = nullptr; cap = 0;
      const size_t want = m + m / 4 + 64;
      if (cudaHostAlloc((void**)&p, want * sizeof(T), cudaHostAllocDefault) != cudaSuccess) { p = nullptr; n = 0; return false; }
      cap = want;
    }
    n = m;
    return true;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; cap = n = 0; }
  T& operator[](size_t i) { return p[i]; }
  T* data() { return p; }
  T& back() { return p[n - 1]; }
};

struct KTime { const char* name; cudaEvent_t a, b; float ms; };

// Certified verdict of the genotype model at a pure position (computed from hm_params by
// make_norm_cert; k_norm_bits receives n_min and the table thr derived from it).  With n reads
// of the reference allele r and qualities b_i:
//   PL_rr     = -10 (M0 + lp_homref)        M0 = sum lut_hom[b_i]
//   PL_het    = -10 (M1 + lp_het)           M1 = sum lut_het[b_i]   (= M0 - n log10 2 up to 1e-13)
//   PL_hetalt = -10 (M2 + lp_hetalt)        M2 = sum lut_err[b_i]   (= -sum b_i / 30 up to 1e-13)
//   PL_homalt = -10 (M2 + lp_homalt)
// every other genotype equals one of these four (adding exact zeros is exact).  Homref is the
// argmin and GQ = int(second - best) >= min_gq iff both differences are >= max(min_gq, 0) and > 0:
//   PL_het - PL_rr      = 10 n log10 2 + 10 (lp_homref - lp_het)                    -> n >= n_min
//   PL_other - PL_rr   >= 10 (sum b_i / 30 - f1 * x / 254) + 10 (lp_homref - max(lp_hetalt, lp_homalt))
//     with x = min(254 n, 255 n - sum b_i), f1 = -lut_hom[1]: -lut_hom is convex and decreasing,
//     so -M0 <= f1 * (255 n - sum b_i) / 254 and trivially <= f1 * n  (all b_i >= 1).
// `margin` keeps the comparison away from the fp64 rounding of the reference's own sums (1e-9 at
// most for depth <= 255); a position that fails the test is simply evaluated exactly.
struct NormCert {
  int32_t enabled;
  int32_t n_min;       // smallest depth whose het - homref difference is certified
  double a_bq;         // 10 / 30
  double a_x;          // 10 * f1 / 254
  double c_oth;        // 10 (lp_homref - max(lp_hetalt, lp_homalt))
  double need;         // max(min_gq, 0) + margin
  long long ia_bq, ia_x, i_need; // floor(a_bq 2^20), ceil(a_x 2^20), ceil((need - c_oth) 2^20)
};

}  // namespace

struct hm_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  std::string err;
  bool have_params = false, have_batch = false;
  hm_params params;
  DevParams dp;
  // resident batch
  uint64_t n_reads = 0, n_ops_total = 0, seq_bytes = 0, bq_bytes = 0;
  uint32_t max_qname_id = 0;
  PinVec<int32_t> h_pmax;
  bool upload_pending = false;  // hm_upload_batch_compact_begin: the copies of the last upload have not been waited for
  DevBuf b_tstart, b_tend, b_qstart, b_qlen, b_mapq, b_flags, b_qname, b_seq_off, b_bq_off, b_op_off, b_n_ops,
      b_seq, b_bq, b_ops, b_op_t, b_op_q, b_mm, b_bq_total, b_n_match, b_n_sub, b_ins_len, b_del_len, b_n_mm, b_gate,
      b_pmax;
  DevBatch db;
  // sets / phase
  DevBuf b_common, b_pon, b_hpos, b_href, b_halt, b_hbit, b_set_off;
  DevSets dsets = {nullptr, 0, nullptr, 0};
  DevPhase dphase = {nullptr, nullptr, nullptr, nullptr, nullptr, 0};
  // work buffers
  DevBuf b_chunks, b_pair_off, b_pair_hap, b_qseen, b_keys, b_keys_sorted, b_cub, b_records, b_counters;
  DevBuf b_ref, b_norm_out, b_lut, b_tile_off, b_agg, b_geom, b_bidx, b_brecs;
  cudaStream_t copy_stream = nullptr;       // record read-back runs here so it can overlap the next call's kernels
  cudaEvent_t ev_copy_done[2] = {nullptr, nullptr};
  DevBuf b_records_alt;                     // second record buffer: calls alternate
  DevBuf b_compact[2], b_keep, b_kpos, b_bpos; // HM_OPT_OMIT_RESTATEMENTS: compacted records, keep flags, their scan
  bool omit_restatements = false;
  int rec_parity = 0;
  bool copy_pending = false;
  struct PendingCopy { void* dst; const void* src; size_t bytes; };
  std::vector<PendingCopy> deferred;        // record copies of the last async call, not enqueued yet
  int deferred_parity = 0;
  cudaEvent_t ev_go = nullptr;              // recorded after k_read_scan: the deferred copies start behind it
  cudaEvent_t ev_up = nullptr;              // recorded behind the last host -> device copy of an upload
  unsigned long long* h_cnt_pin = nullptr; // pinned: counters + boundary indices + boundary records of a call
  DevLut dlut = {nullptr};
  // pinned staging for records coming back, final records of the last call
  hm_site_record* h_stage = nullptr;
  size_t h_stage_cap = 0;
  std::vector<hm_site_record> final_recs;
  // timing
  std::vector<KTime> ktimes;
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  float last_total_ms = 0.f;
  int last_launches = 0;
  size_t ref_len = 0; // length of the contig left resident by hm_set_reference (0: none)
  NormCert cert;      // certified-verdict constants of the normcounts bit-vector pass
  unsigned long long last_norm_sites = 0; // positions the last normcounts call evaluated exactly
  DevBuf b_push, b_span_cnt; // k_norm_bits: 32 site words and a site count per span
  DevBuf b_sites, b_koff, b_tile_info, b_edge_counts, b_edge_hpos, b_edge_href, b_bqmask, b_bqexc, b_bqexc_off;
  uint64_t edge_n = 0;
  uint32_t edge_band = 0;
  // fused call path
  std::vector<uint64_t> h_ops_prefix;       // ops of the reads before read r (candidate slots a chunk can need)
  std::vector<uint8_t> h_named;             // scratch of the shared-query-name test of an upload
  uint32_t site_slots = HM_SITE_SLOTS;      // entry slots per site of the fused call path: about twice the batch's mean depth
  bool dup_names = false;                   // two primary records of the resident batch share a query name
  int call_path = 0;                        // hm_last_call_path
  bool ktiming = true;                      // HM_OPT_KERNEL_TIMING: CUDA events around the kernels of a call
  bool own_launch_count = false;            // last_launches was counted launch by launch (fused path)
  uint64_t site_cap_hint = 0;               // high-water mark of distinct sites per call
  char* h_geom_pin = nullptr;
  size_t h_geom_cap = 0;
  struct Pending { bool active = false; std::vector<hm_chunk> chunks; uint64_t site_cap = 0; size_t bcap = 0; int n_launched = 0, parity = 0; bool omit = false; } pend;
  DevBuf b_cgeom, b_seg_keys, b_seg_read, b_keys_tmp, b_gscratch, b_czero, b_tiles, b_pair_c;
  // bit-vector normcounts path (normbits.cuh)
  PinVec<uint32_t> h_cw_off;                // per read: first word of its cal bit vector
  uint64_t n_cw = 0;                        // words of all cal bit vectors (>= 2^32: the path is not used)
  uint16_t cert_thr[256];                   // smallest callable count that certifies a pure position of depth n (0xffff: none)
  uint64_t packed_pos = 0;                  // positions b_ref2 / b_tri8 cover for the reference now in b_ref (0: not packed)
  DevBuf b_cw_off, b_calw, b_impure, b_ref2, b_tri8, b_thr, b_span_off, b_exc_minmax, b_sdiff, b_cal_ok;
  bool compact_resident = false;            // the resident batch came as bitmap + exceptions: both are still on the device
  uint32_t modal = 0;
  // device BAM decoder (hm_decode_bam_*, bamgpu.cuh)
  DevBuf b_comp, b_pcoff, b_pcsize, b_pisize, b_puoff, b_pcrc, b_pentry, b_inflated, b_blk_code, b_derr, b_seg_cnt,
      b_seg_off, b_recoff, b_recinfo, b_cnt, b_scan, b_ecode, b_earg, b_names, b_name_off;
  PinVec<int32_t> hd_tstart, hd_tend, hd_qstart, hd_qlen;   // per-read arrays of the last hm_decode_bam_begin
  PinVec<uint32_t> hd_n_ops;
  PinVec<uint64_t> hd_bq_off, hd_op_off, hd_name_off, hd_seq_off, hd_scal; // hd_scal: walk / scan totals read back
  PinVec<char> hd_names;
  PinVec<bamgpu::Err> hd_err;
  std::vector<uint8_t> hd_flags;
  uint64_t dec_n = 0, dec_ops = 0, dec_bq = 0, dec_seq = 0;  // dec_seq: base-stream bytes (0: decoded without it)
  bool dec_ready = false;                   // hm_decode_bam_begin succeeded, hm_decode_bam_end has not run
};

namespace {

int fail(hm_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (c) c->err = buf;
  return code;
}
#define CU(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) return fail(ctx, HM_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
  } while (0)

cudaEvent_t next_event(hm_ctx* ctx) {
  if (ctx->ev_used == ctx->ev_pool.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    ctx->ev_pool.push_back(e);
  }
  return ctx->ev_pool[ctx->ev_used++];
}
void t_begin(hm_ctx* ctx, const char* name) {
  if (!ctx->ktiming) return;
  KTime k{name, next_event(ctx), next_event(ctx), 0.f};
  cudaEventRecord(k.a, ctx->stream);
  ctx->ktimes.push_back(k);
}
void t_end(hm_ctx* ctx) { if (ctx->ktiming) cudaEventRecord(ctx->ktimes.back().b, ctx->stream); }
void t_reset(hm_ctx* ctx) { ctx->ktimes.clear(); ctx->ev_used = 0; }
void t_collect(hm_ctx* ctx) {
  ctx->last_total_ms = 0.f;
  if (!ctx->own_launch_count) ctx->last_launches = (int)ctx->ktimes.size();
  for (auto& k : ctx->ktimes) cudaEventElapsedTime(&k.ms, k.a, k.b);
  if (!ctx->ktimes.empty()) cudaEventElapsedTime(&ctx->last_total_ms, ctx->ktimes.front().a, ctx->ktimes.back().b);
}

template <typename T>
int upload(hm_ctx* ctx, DevBuf& buf, const T* src, size_t n, size_t pad_elems = 0) {
  CU(buf.ensure((n + pad_elems) * sizeof(T) + 16));
  if (n) CU(cudaMemcpyAsync(buf.p, src, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  return HM_OK;
}

void make_dev_params(hm_ctx* ctx) {
  const hm_params& p = ctx->params;
  DevParams& d = ctx->dp;
  d.min_qv = p.min_qv; d.min_mapq = p.min_mapq; d.qlen_lower_limit = p.qlen_lower_limit;
  d.qlen_upper_limit = p.qlen_upper_limit; d.min_gq = p.min_gq; d.min_bq = p.min_bq;
  d.max_mismatch_count = p.max_mismatch_count; d.mismatch_window = p.mismatch_window;
  d.min_ref_count = p.min_ref_count; d.min_alt_count = p.min_alt_count; d.min_hap_count = p.min_hap_count;
  d.phase = p.phase; d.non_human_sample = p.non_human_sample; d.create_panel_of_normals = p.create_panel_of_normals;
  d.min_sequence_identity = p.min_sequence_identity; d.min_trim = p.min_trim; d.md_threshold = p.md_threshold;
}

// Constants of the certified homref verdict at pure positions (NormCert above).  The derivation
// assumes the three per-BQ tables are the reference's own (gtlib.py:47-69); that is verified here
// numerically, and the bit-vector pass is switched off for anything else.
void make_norm_cert(hm_ctx* ctx) {
  const hm_params& p = ctx->params;
  NormCert& c = ctx->cert;
  memset(&c, 0, sizeof(c));
  for (int n = 0; n < 256; n++) ctx->cert_thr[n] = 0xffff;
  const double L2 = 0.30102999566398119521; // log10(2)
  const double f1 = -p.lut_hom[1];
  bool ok = p.min_bq >= 1 && p.min_bq <= 128 && p.min_gq <= 99 && f1 > 0.0 && f1 < 1.0;
  for (int bq = 1; bq < 256 && ok; bq++) {
    const double hom = p.lut_hom[bq], het = p.lut_het[bq], err = p.lut_err[bq];
    if (!(hom <= 0.0) || !(fabs(het - (hom - L2)) <= 1e-9) || !(fabs(err + (double)bq / 30.0) <= 1e-9)) ok = false;
    if (!(-hom <= f1 * (double)(255 - bq) / 254.0 + 1e-12)) ok = false; // chord bound of the convex -lut_hom
  }
  for (int k = 0; k < 4 && ok; k++) if (!(p.log10_prior[k] == p.log10_prior[k]) || fabs(p.log10_prior[k]) > 1e6) ok = false;
  if (!ok) return;
  const double margin = 1e-6;
  c.need = (p.min_gq > 0 ? (double)p.min_gq : 0.0) + margin;
  const double c_het = 10.0 * (p.log10_prior[0] - p.log10_prior[1]);
  double n_min = ceil((c.need + margin - c_het) / (10.0 * L2));
  if (n_min < 1.0) n_min = 1.0;
  if (n_min > 1e6) return;
  c.n_min = (int32_t)n_min;
  c.a_bq = 10.0 / 30.0 * (1.0 - 1e-12);
  c.a_x = 10.0 * f1 / 254.0 * (1.0 + 1e-12);
  c.c_oth = 10.0 * (p.log10_prior[0] - std::max(p.log10_prior[2], p.log10_prior[3])) - margin;
  c.ia_bq = (long long)floor(c.a_bq * 1048576.0);
  c.ia_x = (long long)ceil(c.a_x * 1048576.0);
  c.i_need = (long long)ceil((c.need - c.c_oth) * 1048576.0);
  c.enabled = 1;
  // The bit-vector pass (normbits.cuh) knows the depth n and the callable count cal of a pure position, not the sum of
  // its qualities; every callable base has BQ >= min_bq and every other base BQ >= 1, so s1 >= min_bq cal + (n - cal),
  // and the left side of the test above only grows with s1.  thr[n] = the smallest cal that passes it, made
  // non-decreasing in n because the kernel looks it up with an upper bound of n.
  uint16_t run = 0;
  for (int n = 0; n < 256; n++) {
    uint16_t t = 0xffff;
    if (n >= c.n_min) {
      for (int cal = 0; cal <= n; cal++) {
        const long long s1 = (long long)p.min_bq * cal + (n - cal);
        const long long x = std::min(254ll * n, 255ll * n - s1);
        if (s1 * c.ia_bq - x * c.ia_x >= c.i_need) { t = (uint16_t)cal; break; }
      }
      if (t < run) t = run;
      run = t;
    }
    ctx->cert_thr[n] = t;
  }
}

// The record copies of an asynchronous call are enqueued late, behind the *next* call's sort (past k_read_scan, the
// one HBM-bound kernel of the path, and past the latency-bound candidate / sort kernels a concurrent copy slows most),
// so they overlap its site kernels; without a next call (or when it has no candidates),
// hm_records_wait enqueues them.  after_main: make the copy stream wait for what the main stream has queued so far.
int flush_deferred(hm_ctx* ctx, bool after_main) {
  if (ctx->deferred.empty()) return HM_OK;
  if (after_main) {
    CU(cudaEventRecord(ctx->ev_go, ctx->stream));
    CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_go, 0));
  }
  for (const auto& c : ctx->deferred) CU(cudaMemcpyAsync(c.dst, c.src, c.bytes, cudaMemcpyDeviceToHost, ctx->copy_stream));
  CU(cudaEventRecord(ctx->ev_copy_done[ctx->deferred_parity], ctx->copy_stream));
  ctx->deferred.clear();
  ctx->copy_pending = true;
  return HM_OK;
}

int check_ready(hm_ctx* ctx, const hm_chunk* chunks, size_t n_chunks) {
  if (!ctx) return HM_ERR_ARG;
  if (!ctx->have_params) return fail(ctx, HM_ERR_STATE, "hm_set_params has not been called");
  if (!ctx->have_batch) return fail(ctx, HM_ERR_STATE, "no resident batch: call hm_upload_batch first");
  if (n_chunks && !chunks) return fail(ctx, HM_ERR_ARG, "chunks is NULL");
  if (n_chunks >= (1ull << 28)) return fail(ctx, HM_ERR_ARG, "too many chunks");
  for (size_t i = 0; i < n_chunks; i++) {
    if (chunks[i].read_lo > chunks[i].read_hi || chunks[i].read_hi > ctx->n_reads)
      return fail(ctx, HM_ERR_ARG, "chunk %zu: read range [%u, %u) outside the batch (%llu reads)", i, chunks[i].read_lo,
                  chunks[i].read_hi, (unsigned long long)ctx->n_reads);
    if (ctx->params.phase && (chunks[i].phase_set < 0 || (uint32_t)chunks[i].phase_set >= ctx->dphase.n_sets))
      return fail(ctx, HM_ERR_ARG, "chunk %zu: phase_set %d is not in the phase table", i, chunks[i].phase_set);
  }
  return HM_OK;
}

// the resident batch's per-read quality sums from its one-byte-per-base stream (a compact upload has k_bq_expand)
int launch_bq_sum(hm_ctx* ctx) {
  if (ctx->n_reads == 0) return HM_OK;
  t_reset(ctx);
  t_begin(ctx, "k_bq_sum");
  k_bq_sum<<<(unsigned)((ctx->n_reads * 32 + 255) / 256), 256, 0, ctx->stream>>>(ctx->db);
  t_end(ctx);
  CU(cudaGetLastError());
  return HM_OK;
}

// k_read_scan over the resident batch
int launch_read_scan(hm_ctx* ctx) {
  if (ctx->n_reads == 0) return HM_OK;
  const unsigned blocks = (unsigned)((ctx->n_reads * 32 + 255) / 256);
  t_begin(ctx, "k_read_scan");
  k_read_scan<<<blocks, 256, 0, ctx->stream>>>(ctx->db, ctx->dp);
  t_end(ctx);
  CU(cudaGetLastError());
  return HM_OK;
}

int upload_chunks(hm_ctx* ctx, const hm_chunk* chunks, size_t n_chunks, std::vector<uint64_t>& pair_off) {
  pair_off.assign(n_chunks + 1, 0);
  for (size_t i = 0; i < n_chunks; i++) pair_off[i + 1] = pair_off[i] + (chunks[i].read_hi - chunks[i].read_lo);
  int rc = upload(ctx, ctx->b_chunks, chunks, n_chunks);
  if (rc) return rc;
  return upload(ctx, ctx->b_pair_off, pair_off.data(), pair_off.size());
}

}  // namespace

extern "C" {

int hm_abi_version(void) { return HM_ABI_VERSION; }

int hm_device_count(void) {
  int n = 0;
  return cudaGetDeviceCount(&n) == cudaSuccess ? n : 0;
}

size_t hm_abi_sizeof(int which) {
  switch (which) {
    case 0: return sizeof(hm_read_batch);
    case 1: return sizeof(hm_chunk);
    case 2: return sizeof(hm_params);
    case 3: return sizeof(hm_site_record);
    case 4: return sizeof(hm_bq_compact);
    case 5: return sizeof(hm_bgzf_plan);
    default: return 0;
  }
}

int hm_create(int cuda_device, hm_ctx** out) {
  if (!out) return HM_ERR_ARG;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || cuda_device < 0 || cuda_device >= n) return HM_ERR_NO_DEVICE;
  if (cudaSetDevice(cuda_device) != cudaSuccess) return HM_ERR_NO_DEVICE;
  hm_ctx* ctx = new hm_ctx();
  ctx->device = cuda_device;
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete ctx;
    return HM_ERR_CUDA;
  }
  memset(&ctx->db, 0, sizeof(ctx->db));
  if (cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_copy_done[0], cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_copy_done[1], cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_go, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_up, cudaEventDisableTiming | cudaEventBlockingSync) != cudaSuccess) {
    delete ctx;
    return HM_ERR_CUDA;
  }
  *out = ctx;
  return HM_OK;
}

void hm_destroy(hm_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream); // also ends an upload that was not waited for
  if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
  for (cudaEvent_t e : ctx->ev_copy_done) if (e) cudaEventDestroy(e);
  if (ctx->ev_go) cudaEventDestroy(ctx->ev_go);
  if (ctx->ev_up) cudaEventDestroy(ctx->ev_up);
  ctx->b_records_alt.release();
  ctx->b_compact[0].release(); ctx->b_compact[1].release(); ctx->b_keep.release(); ctx->b_kpos.release(); ctx->b_bpos.release();
  DevBuf* bufs[] = {&ctx->b_tstart, &ctx->b_tend, &ctx->b_qstart, &ctx->b_qlen, &ctx->b_mapq, &ctx->b_flags, &ctx->b_qname,
                    &ctx->b_seq_off, &ctx->b_bq_off, &ctx->b_op_off, &ctx->b_n_ops, &ctx->b_seq, &ctx->b_bq, &ctx->b_ops,
                    &ctx->b_op_t, &ctx->b_op_q, &ctx->b_mm, &ctx->b_bq_total, &ctx->b_n_match, &ctx->b_n_sub,
                    &ctx->b_ins_len, &ctx->b_del_len, &ctx->b_n_mm, &ctx->b_gate, &ctx->b_pmax, &ctx->b_common, &ctx->b_pon,
                    &ctx->b_hpos, &ctx->b_href, &ctx->b_halt, &ctx->b_hbit, &ctx->b_set_off, &ctx->b_chunks,
                    &ctx->b_pair_off, &ctx->b_pair_hap, &ctx->b_qseen, &ctx->b_keys, &ctx->b_keys_sorted, &ctx->b_cub,
                    &ctx->b_records, &ctx->b_counters, &ctx->b_ref, &ctx->b_norm_out, &ctx->b_lut, &ctx->b_tile_off, &ctx->b_agg, &ctx->b_geom, &ctx->b_bidx, &ctx->b_brecs, &ctx->b_sites, &ctx->b_push, &ctx->b_span_cnt, &ctx->b_koff, &ctx->b_tile_info, &ctx->b_edge_counts, &ctx->b_edge_hpos, &ctx->b_edge_href, &ctx->b_bqmask, &ctx->b_bqexc, &ctx->b_bqexc_off,
                    &ctx->b_cgeom, &ctx->b_seg_keys, &ctx->b_seg_read, &ctx->b_keys_tmp, &ctx->b_gscratch, &ctx->b_czero, &ctx->b_tiles, &ctx->b_pair_c,
                    &ctx->b_cw_off, &ctx->b_calw, &ctx->b_impure, &ctx->b_ref2, &ctx->b_tri8, &ctx->b_thr, &ctx->b_span_off, &ctx->b_exc_minmax, &ctx->b_sdiff, &ctx->b_cal_ok,
                    &ctx->b_comp, &ctx->b_pcoff, &ctx->b_pcsize, &ctx->b_pisize, &ctx->b_puoff, &ctx->b_pcrc, &ctx->b_pentry, &ctx->b_inflated,
                    &ctx->b_blk_code, &ctx->b_derr, &ctx->b_seg_cnt, &ctx->b_seg_off, &ctx->b_recoff, &ctx->b_recinfo, &ctx->b_cnt,
                    &ctx->b_scan, &ctx->b_ecode, &ctx->b_earg, &ctx->b_names, &ctx->b_name_off};
  for (DevBuf* b : bufs) b->release();
  if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
  if (ctx->h_cnt_pin) cudaFreeHost(ctx->h_cnt_pin);
  if (ctx->h_geom_pin) cudaFreeHost(ctx->h_geom_pin);
  ctx->h_pmax.release(); ctx->h_cw_off.release();
  ctx->hd_tstart.release(); ctx->hd_tend.release(); ctx->hd_qstart.release(); ctx->hd_qlen.release(); ctx->hd_n_ops.release();
  ctx->hd_bq_off.release(); ctx->hd_op_off.release(); ctx->hd_name_off.release(); ctx->hd_seq_off.release(); ctx->hd_scal.release(); ctx->hd_names.release();
  ctx->hd_err.release();
  for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* hm_last_error(const hm_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

/* run the context's work on a caller-owned CUDA stream (cudaStream_t as void*), so that
 * the caller's own events bracket it; NULL restores the private stream */
int hm_set_stream(hm_ctx* ctx, void* cuda_stream) {
  if (!ctx) return HM_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  if (cuda_stream) { ctx->stream = (cudaStream_t)cuda_stream; ctx->own_stream = false; }
  else { CU(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)); ctx->own_stream = true; }
  return HM_OK;
}

/* page-lock / unlock caller memory so the H2D copies of hm_upload_batch run at PCIe speed */
int hm_host_register(hm_ctx* ctx, void* p, size_t bytes) {
  if (!ctx || !p) return HM_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  CU(cudaHostRegister(p, bytes, cudaHostRegisterDefault));
  return HM_OK;
}
int hm_host_unregister(hm_ctx* ctx, void* p) {
  if (!ctx || !p) return HM_ERR_ARG;
  CU(cudaHostUnregister(p));
  return HM_OK;
}

int hm_set_params(hm_ctx* ctx, const hm_params* params) {
  if (!ctx || !params) return HM_ERR_ARG;
  if (params->mismatch_window < 0 || params->qlen_upper_limit < 0) return fail(ctx, HM_ERR_ARG, "negative window / qlen limit");
  CU(cudaSetDevice(ctx->device));
  ctx->params = *params;
  make_dev_params(ctx);
  make_norm_cert(ctx);
  DevTables t;
  memcpy(t.lut[0], params->lut_hom, sizeof(t.lut[0]));
  memcpy(t.lut[1], params->lut_het, sizeof(t.lut[1]));
  memcpy(t.lut[2], params->lut_err, sizeof(t.lut[2]));
  memcpy(t.log10_prior, params->log10_prior, sizeof(t.log10_prior));
  CU(cudaStreamSynchronize(ctx->stream));
  CU(cudaMemcpyToSymbol(c_tab, &t, sizeof(t)));
  CU(ctx->b_lut.ensure(sizeof(t.lut)));
  CU(cudaMemcpy(ctx->b_lut.p, t.lut, sizeof(t.lut), cudaMemcpyHostToDevice));
  ctx->dlut.lut = ctx->b_lut.as<double>();
  ctx->have_params = true;
  return HM_OK;
}

int hm_set_site_sets(hm_ctx* ctx, const uint64_t* common_sorted, size_t n_common, const uint64_t* pon_sorted, size_t n_pon) {
  if (!ctx) return HM_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  for (size_t i = 1; i < n_common; i++) if (common_sorted[i - 1] > common_sorted[i]) return fail(ctx, HM_ERR_ARG, "common-SNP keys are not sorted");
  for (size_t i = 1; i < n_pon; i++) if (pon_sorted[i - 1] > pon_sorted[i]) return fail(ctx, HM_ERR_ARG, "panel-of-normals keys are not sorted");
  int rc = upload(ctx, ctx->b_common, common_sorted, n_common);
  if (rc) return rc;
  rc = upload(ctx, ctx->b_pon, pon_sorted, n_pon);
  if (rc) return rc;
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->dsets = DevSets{ctx->b_common.as<uint64_t>(), n_common, ctx->b_pon.as<uint64_t>(), n_pon};
  return HM_OK;
}

int hm_set_phase_sets(hm_ctx* ctx, const int32_t* hpos, const uint8_t* href, const uint8_t* halt, const uint8_t* hbit,
                      size_t n_hetsnp, const uint64_t* set_off, size_t n_sets) {
  if (!ctx) return HM_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  if (n_sets && (!set_off || set_off[n_sets] != n_hetsnp)) return fail(ctx, HM_ERR_ARG, "set_off[n_sets] must equal n_hetsnp");
  for (size_t s = 0; s < n_sets; s++) {
    if (set_off[s] > set_off[s + 1]) return fail(ctx, HM_ERR_ARG, "set_off is not ascending");
    for (uint64_t k = set_off[s] + 1; k < set_off[s + 1]; k++)
      if (hpos[k - 1] > hpos[k]) return fail(ctx, HM_ERR_ARG, "hpos is not ascending inside phase set %zu", s);
  }
  int rc;
  if ((rc = upload(ctx, ctx->b_hpos, hpos, n_hetsnp))) return rc;
  if ((rc = upload(ctx, ctx->b_href, href, n_hetsnp))) return rc;
  if ((rc = upload(ctx, ctx->b_halt, halt, n_hetsnp))) return rc;
  if ((rc = upload(ctx, ctx->b_hbit, hbit, n_hetsnp))) return rc;
  if ((rc = upload(ctx, ctx->b_set_off, set_off, n_sets ? n_sets + 1 : 0))) return rc;
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->dphase = DevPhase{ctx->b_hpos.as<int32_t>(), ctx->b_href.as<uint8_t>(), ctx->b_halt.as<uint8_t>(),
                         ctx->b_hbit.as<uint8_t>(), ctx->b_set_off.as<uint64_t>(), (uint32_t)n_sets};
  return HM_OK;
}

static int upload_batch_impl(hm_ctx* ctx, const hm_read_batch* b, const hm_bq_compact* cq, bool wait = true);

int hm_upload_batch(hm_ctx* ctx, const hm_read_batch* b) { return upload_batch_impl(ctx, b, nullptr); }

int hm_upload_batch_compact(hm_ctx* ctx, const hm_read_batch* b, const hm_bq_compact* cq) {
  if (!cq) return HM_ERR_ARG;
  return upload_batch_impl(ctx, b, cq);
}

/* hm_upload_batch_compact that returns as soon as its copies are enqueued: the caller's buffers must stay as they are
 * until hm_upload_wait (or the next hm_upload_* / hm_destroy of the context) has returned.  Calls may be enqueued on the
 * context meanwhile (they run behind the copies).  A worker that alternates two contexts enqueues the upload of group
 * k + 1 on one before it waits for the upload of group k on the other, so the copy engine never idles between them. */
int hm_upload_batch_compact_begin(hm_ctx* ctx, const hm_read_batch* b, const hm_bq_compact* cq) {
  if (!cq) return HM_ERR_ARG;
  return upload_batch_impl(ctx, b, cq, false);
}
int hm_upload_wait(hm_ctx* ctx) {
  if (!ctx) return HM_ERR_ARG;
  if (ctx->upload_pending) {
    CU(cudaSetDevice(ctx->device));
    CU(cudaEventSynchronize(ctx->ev_up));
    ctx->upload_pending = false;
  }
  return HM_OK;
}

// The O(reads) checks of a batch on the host and the tables derived from it (running maximum of tend,
// cal-word offsets, op prefix, shared query names, entry slots per site), for both ways a batch becomes resident
// (hm_upload_batch*, hm_decode_bam_end).  A batch that fails is never used; the stream is waited for before the error
// returns, so the caller may free its buffers.
static int batch_tables(hm_ctx* ctx, const hm_read_batch* b, const hm_bq_compact* cq, bool has_seq) {
  const uint64_t n = b->n_reads;
#define BAD(...) do { cudaStreamSynchronize(ctx->stream); return fail(ctx, HM_ERR_ARG, __VA_ARGS__); } while (0)
  // structural validation (cheap, O(reads)); the kernels binary-search on these invariants
  if (!ctx->h_pmax.resize(n) || !ctx->h_cw_off.resize(n + 1)) BAD("out of page-locked host memory for %llu reads", (unsigned long long)n);
  uint64_t n_cw = 0, span_sum = 0;
  int32_t run = INT32_MIN;
  uint32_t max_q = 0;
  for (uint64_t r = 0; r < n; r++) {
    if (r && b->tstart[r] < b->tstart[r - 1]) BAD("read %llu: batch is not sorted by reference_start", (unsigned long long)r);
    if (b->tend[r] < b->tstart[r] || b->qlen[r] <= 0 || b->qstart[r] < 0 || b->qstart[r] > b->qlen[r])
      BAD("read %llu: inconsistent coordinates", (unsigned long long)r);
    if ((has_seq && (b->seq_off[r] & 15)) || (b->bq_off[r] & 15)) BAD("read %llu: seq_off / bq_off not 16-byte aligned", (unsigned long long)r);
    if (b->bq_off[r] + (uint64_t)b->qlen[r] > b->bq_bytes || (has_seq && b->seq_off[r] + ((uint64_t)b->qlen[r] + 3) / 4 > b->seq_bytes) ||
        b->op_off[r] + b->n_ops[r] > b->n_ops_total)
      BAD("read %llu: offsets outside the buffers", (unsigned long long)r);
    if (cq && (cq->exc_off[r] > cq->exc_off[r + 1] || cq->exc_off[r + 1] > cq->exc_bytes || cq->exc_off[r + 1] - cq->exc_off[r] > (uint64_t)b->qlen[r]))
      BAD("read %llu: hm_bq_compact.exc_off is inconsistent", (unsigned long long)r);
    if (b->tend[r] > run) run = b->tend[r];
    span_sum += (uint64_t)(b->tend[r] - b->tstart[r]);
    ctx->h_pmax[r] = run;
    ctx->h_cw_off[r] = (uint32_t)n_cw;
    if (b->tend[r] > b->tstart[r] && b->tstart[r] >= 0) n_cw += (uint64_t)(((b->tend[r] - 1) >> 5) - (b->tstart[r] >> 5) + 1);
    if (b->qname_id[r] > max_q) max_q = b->qname_id[r];
  }
  ctx->max_qname_id = max_q;
  { // entry slots per site: a site's file-order read range holds about `depth` reads; twice the mean depth (64 at least,
    // 512 at most, a multiple of 32) keeps all but the deepest pileups out of k_site_reduce's own op walk
    const double covered = n ? (double)std::max<int64_t>((int64_t)run - (int64_t)b->tstart[0], 1) : 1.0;
    const double depth = (double)span_sum / covered;
    uint32_t slots = (uint32_t)std::min(512.0, std::max(64.0, 2.0 * depth));
    slots = (slots + 31u) & ~31u;
    if (const char* e = getenv("HIMUT_B200_SITE_SLOTS")) slots = (uint32_t)std::min(512, std::max(1, atoi(e))); // tests: force the deep-pileup walk
    ctx->site_slots = slots;
  }
  // candidate slots a chunk can need = ops of the reads it fetches; shared query names among primary records
  // (the phase check of a site then goes by name, caller.py:556-567)
  ctx->h_ops_prefix.resize(n + 1);
  ctx->h_ops_prefix[0] = 0;
  ctx->dup_names = false;
  {
    ctx->h_named.assign((size_t)max_q + 1, 0);
    uint8_t* named = ctx->h_named.data();
    for (uint64_t r = 0; r < n; r++) {
      ctx->h_ops_prefix[r + 1] = ctx->h_ops_prefix[r] + b->n_ops[r];
      if (b->flags[r] & HM_READ_SECONDARY) continue;
      if (named[b->qname_id[r]]) ctx->dup_names = true;
      named[b->qname_id[r]] = 1;
    }
  }
  if (b->n_reads && b->tstart[0] < 0) BAD("negative reference_start");
#undef BAD
  ctx->h_cw_off[n] = (uint32_t)n_cw;
  ctx->n_cw = n_cw;
  return HM_OK;
}

// the derived tables to the device and the resident batch's device view (the per-read arrays are in place)
static int bind_batch(hm_ctx* ctx, const hm_read_batch* b, bool has_seq) {
  const uint64_t n = b->n_reads;
  int rc;
  if ((rc = upload(ctx, ctx->b_pmax, ctx->h_pmax.data(), n))) return rc;
  if (ctx->n_cw < (1ull << 32) && (rc = upload(ctx, ctx->b_cw_off, ctx->h_cw_off.data(), n + 1))) return rc;
  const size_t no = (size_t)b->n_ops_total;
  CU(ctx->b_op_t.ensure(no * 4 + 16)); CU(ctx->b_op_q.ensure(no * 4 + 16)); CU(ctx->b_mm.ensure(no * 4 + 16));
  CU(ctx->b_bq_total.ensure(n * 8 + 16)); CU(ctx->b_n_match.ensure(n * 4 + 16)); CU(ctx->b_n_sub.ensure(n * 4 + 16));
  CU(ctx->b_ins_len.ensure(n * 4 + 16)); CU(ctx->b_del_len.ensure(n * 4 + 16)); CU(ctx->b_n_mm.ensure(n * 4 + 16));
  CU(ctx->b_gate.ensure(n + 16));
  DevBatch& d = ctx->db;
  d.n_reads = n;
  d.tstart = ctx->b_tstart.as<int32_t>(); d.tend = ctx->b_tend.as<int32_t>(); d.qstart = ctx->b_qstart.as<int32_t>();
  d.qlen = ctx->b_qlen.as<int32_t>(); d.mapq = ctx->b_mapq.as<uint8_t>(); d.flags = ctx->b_flags.as<uint8_t>();
  d.qname_id = ctx->b_qname.as<uint32_t>(); d.seq_off = has_seq ? ctx->b_seq_off.as<uint64_t>() : nullptr; d.bq_off = ctx->b_bq_off.as<uint64_t>();
  d.op_off = ctx->b_op_off.as<uint64_t>(); d.n_ops = ctx->b_n_ops.as<uint32_t>(); d.seq = has_seq ? ctx->b_seq.as<uint8_t>() : nullptr;
  d.bq = ctx->b_bq.as<uint8_t>(); d.ops = ctx->b_ops.as<uint32_t>();
  d.op_t = ctx->b_op_t.as<uint32_t>(); d.op_q = ctx->b_op_q.as<uint32_t>(); d.mm_pos = ctx->b_mm.as<int32_t>();
  d.bq_total = ctx->b_bq_total.as<unsigned long long>(); d.n_match = ctx->b_n_match.as<int32_t>();
  d.n_sub = ctx->b_n_sub.as<int32_t>(); d.ins_len = ctx->b_ins_len.as<int32_t>(); d.del_len = ctx->b_del_len.as<int32_t>();
  d.n_mm = ctx->b_n_mm.as<int32_t>(); d.gate = ctx->b_gate.as<uint8_t>(); d.pmax_tend = ctx->b_pmax.as<int32_t>();
  ctx->n_reads = n; ctx->n_ops_total = b->n_ops_total; ctx->seq_bytes = b->seq_bytes; ctx->bq_bytes = b->bq_bytes;
  return HM_OK;
}

static int upload_batch_impl(hm_ctx* ctx, const hm_read_batch* b, const hm_bq_compact* cq, bool wait) {
  if (!ctx || !b) return HM_ERR_ARG;
  if (!cq && !b->bq) return fail(ctx, HM_ERR_ARG, "batch has no quality stream");
  // seq == NULL: no base stream.  The bases of match runs are then the reference allele of the site that asks
  // (what a cs match means, cslib.py:22-29); substituted bases travel in the ops.  `call` and the phase edges
  // need nothing else; normcounts does (for now) and refuses such a batch.
  const bool has_seq = b->seq != nullptr;
  if (!has_seq && b->seq_bytes) return fail(ctx, HM_ERR_ARG, "seq is NULL but seq_bytes is not 0");
  if (has_seq && !b->seq_off) return fail(ctx, HM_ERR_ARG, "seq without seq_off");
  if (cq) {
    if (!cq->mask || !cq->exc_off || (cq->exc_bytes && !cq->exc)) return fail(ctx, HM_ERR_ARG, "incomplete hm_bq_compact");
    if (cq->mask_bytes * 8 != b->bq_bytes) return fail(ctx, HM_ERR_ARG, "hm_bq_compact.mask_bytes must be bq_bytes / 8");
  }
  CU(cudaSetDevice(ctx->device));
  if (ctx->upload_pending) { // an upload that was not waited for: its copies still read the page-locked tables rewritten below
    CU(cudaEventSynchronize(ctx->ev_up));
    ctx->upload_pending = false;
  }
  ctx->have_batch = false;
  const uint64_t n = b->n_reads;
  if (n >= (1ull << 32)) return fail(ctx, HM_ERR_ARG, "too many reads in one batch");
  if ((b->seq_bytes & 15) || (b->bq_bytes & 15)) return fail(ctx, HM_ERR_ARG, "seq / bq buffers must be padded to 16 bytes");
  // The large streams leave first (copy engine, in stream order); the O(reads) validation below runs on the host while
  // they move.  A batch that fails it is never used (have_batch stays false); the copies are waited for before the
  // error is returned, so the caller may free its buffers.
  int rc;
#define UP(buf, field, count) if ((rc = upload(ctx, ctx->buf, b->field, (size_t)(count)))) return rc
  if (cq) {
    if ((rc = upload(ctx, ctx->b_bqmask, cq->mask, (size_t)cq->mask_bytes))) return rc;
    if ((rc = upload(ctx, ctx->b_bqexc, cq->exc, (size_t)cq->exc_bytes, 16))) return rc;
  } else { UP(b_bq, bq, b->bq_bytes); }
  if (has_seq) { UP(b_seq, seq, b->seq_bytes); }
  UP(b_ops, ops, b->n_ops_total);
  if ((rc = batch_tables(ctx, b, cq, has_seq))) return rc;
  UP(b_tstart, tstart, n); UP(b_tend, tend, n); UP(b_qstart, qstart, n); UP(b_qlen, qlen, n);
  UP(b_mapq, mapq, n); UP(b_flags, flags, n); UP(b_qname, qname_id, n);
  UP(b_bq_off, bq_off, n); UP(b_op_off, op_off, n); UP(b_n_ops, n_ops, n);
  if (has_seq) { UP(b_seq_off, seq_off, n); }
  if (cq) {
    CU(ctx->b_bq.ensure(b->bq_bytes + 16));
    if ((rc = upload(ctx, ctx->b_bqexc_off, cq->exc_off, (size_t)n + 1))) return rc;
  }
#undef UP
  if ((rc = bind_batch(ctx, b, has_seq))) return rc;
  ctx->compact_resident = false;
  CU(cudaEventRecord(ctx->ev_up, ctx->stream)); // every host buffer has been read once this fires
  if (cq && n) {
    CU(ctx->b_exc_minmax.ensure(2 * n + 16));
    ctx->modal = (uint32_t)cq->modal;
    ctx->compact_resident = true;
    t_reset(ctx);
    t_begin(ctx, "k_bq_expand");
    k_bq_expand<<<(unsigned)((n * 32 + 255) / 256), 256, 0, ctx->stream>>>(ctx->db, ctx->b_bqmask.as<uint8_t>(), ctx->b_bqexc.as<uint8_t>(),
                                                                         ctx->b_bqexc_off.as<uint64_t>(), (uint32_t)cq->modal, ctx->b_bq.as<uint8_t>(),
                                                                         ctx->b_exc_minmax.as<uint8_t>(), ctx->db.bq_total);
    t_end(ctx);
    CU(cudaGetLastError());
  } else if ((rc = launch_bq_sum(ctx))) return rc;
  if (wait) CU(cudaEventSynchronize(ctx->ev_up)); // the caller may reuse its buffers after return; k_bq_expand may still be running
  ctx->upload_pending = !wait;
  ctx->have_batch = true;
  return HM_OK;
}

// ------------------------------------------------------------------ device BAM decoder (bamgpu.cuh)
// the message of the first failing record (index r of the walk) of the last decode, as the host decoder words it
static int decode_record_error(hm_ctx* ctx, const hm_bgzf_plan* pl, unsigned long long r) {
  uint8_t code = 0;
  long long arg = 0;
  bamgpu::RecInfo info;
  CU(cudaMemcpyAsync(&code, ctx->b_ecode.as<uint8_t>() + r, 1, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(&arg, ctx->b_earg.as<long long>() + r, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(&info, ctx->b_recinfo.as<bamgpu::RecInfo>() + r, sizeof(info), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  if (code == 0 || code >= E_N_CODES) return fail(ctx, HM_ERR_ARG, "device BAM decoder: record %llu failed without a code", r);
  if (REC_ERR_ON_PATH(code)) return fail(ctx, HM_ERR_ARG, REC_ERR[code], pl->path ? pl->path : "", (long)arg);
  char name[257];  // the record passed the field checks: its name ends inside it, within 256 bytes
  CU(cudaMemcpyAsync(name, ctx->b_inflated.as<uint8_t>() + info.p + 4 + 32, 256, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  name[256] = 0;
  return fail(ctx, HM_ERR_ARG, REC_ERR[code], name, (long)arg);
}

static int decode_begin_impl(hm_ctx* ctx, const hm_bgzf_plan* pl, int rid, int32_t start, int32_t end, bool want_seq,
                             uint64_t* n_reads) {
  using namespace bamgpu;
  const uint64_t nb = pl->n_blocks, ne = pl->n_entry;
  ctx->dec_n = ctx->dec_ops = 0;
  ctx->dec_bq = 16;
  ctx->dec_seq = want_seq ? 16 : 0;  // the host decoder's empty batch: 16 zero bytes of each stream it has
  if (nb == 0 || ne == 0) return HM_OK;
  // the plan comes from outside: every offset the kernels follow is checked here
  if (!pl->comp || !pl->blk_coff || !pl->blk_csize || !pl->blk_isize || !pl->blk_uoff || !pl->blk_crc || !pl->entry)
    return fail(ctx, HM_ERR_ARG, "incomplete hm_bgzf_plan");
  for (uint64_t i = 0; i < nb; i++)
    if (pl->blk_coff[i] + pl->blk_csize[i] != pl->blk_coff[i + 1] || pl->blk_csize[i] < 20 || pl->blk_isize[i] > 65536 ||
        pl->blk_uoff[i] + pl->blk_isize[i] != pl->blk_uoff[i + 1])
      return fail(ctx, HM_ERR_ARG, "hm_bgzf_plan: block %llu is inconsistent", (unsigned long long)i);
  const uint64_t total = pl->blk_uoff[nb];
  if (pl->blk_coff[0] != 0 || pl->blk_coff[nb] != pl->comp_bytes || pl->blk_uoff[0] != 0 || pl->walk_end > total)
    return fail(ctx, HM_ERR_ARG, "hm_bgzf_plan: the block table does not cover the range");
  for (uint64_t e = 0; e < ne; e++)
    if (pl->entry[e] >= pl->walk_end || (e && pl->entry[e] <= pl->entry[e - 1]))
      return fail(ctx, HM_ERR_ARG, "hm_bgzf_plan: entry point %llu is out of order", (unsigned long long)e);
  int rc;
  t_begin(ctx, "h2d_compressed");
  if ((rc = upload(ctx, ctx->b_comp, pl->comp, pl->comp_bytes))) return rc;
  t_end(ctx);
  if ((rc = upload(ctx, ctx->b_pcoff, pl->blk_coff, nb + 1))) return rc;
  if ((rc = upload(ctx, ctx->b_pcsize, pl->blk_csize, nb))) return rc;
  if ((rc = upload(ctx, ctx->b_pisize, pl->blk_isize, nb))) return rc;
  if ((rc = upload(ctx, ctx->b_puoff, pl->blk_uoff, nb + 1))) return rc;
  if ((rc = upload(ctx, ctx->b_pcrc, pl->blk_crc, nb))) return rc;
  if ((rc = upload(ctx, ctx->b_pentry, pl->entry, ne))) return rc;
  CU(ctx->b_inflated.ensure(total + 64));  // 64 zero bytes past the end: the fixed part of a short last record reads there
  CU(cudaMemsetAsync(ctx->b_inflated.as<uint8_t>() + total, 0, 64, ctx->stream));
  CU(ctx->b_blk_code.ensure(nb));
  CU(ctx->b_derr.ensure(sizeof(Err)));
  CU(cudaMemsetAsync(ctx->b_derr.p, 0xff, sizeof(Err), ctx->stream));
  if (!ctx->hd_err.resize(1) || !ctx->hd_scal.resize(5)) return fail(ctx, HM_ERR_ARG, "out of page-locked host memory");
  Err* derr = ctx->b_derr.as<Err>();
  Err& herr = ctx->hd_err[0];
  // inflate: one block per warp (bamgpu.cuh says why)
  const uint64_t per_cta = 1;
  const Plan dpl{ctx->b_comp.as<uint8_t>(), ctx->b_pcoff.as<uint64_t>(), ctx->b_pcsize.as<uint32_t>(), ctx->b_pisize.as<uint32_t>(),
                 ctx->b_puoff.as<uint64_t>(), ctx->b_pcrc.as<uint32_t>(), nb};
  t_begin(ctx, "k_bgzf_inflate");
  k_bgzf_inflate<<<(unsigned)((nb + per_cta - 1) / per_cta), 32, 0, ctx->stream>>>(dpl, ctx->b_inflated.as<uint8_t>(), (uint32_t)per_cta,
                                                                                ctx->b_blk_code.as<uint8_t>(), derr);
  t_end(ctx);
  CU(cudaGetLastError());
  // walk: records per segment, their scan, then the offsets
  CU(ctx->b_seg_cnt.ensure((ne + 1) * 8));
  CU(ctx->b_seg_off.ensure((ne + 1) * 8));
  CU(cudaMemsetAsync(ctx->b_seg_cnt.as<unsigned long long>() + ne, 0, 8, ctx->stream));
  const uint8_t* buf = ctx->b_inflated.as<uint8_t>();
  t_begin(ctx, "k_bam_walk");
  k_bam_walk<<<(unsigned)((ne + 127) / 128), 128, 0, ctx->stream>>>(buf, ctx->b_pentry.as<uint64_t>(), ne, pl->walk_end,
                                                                     ctx->b_seg_cnt.as<unsigned long long>(), nullptr, nullptr, derr);
  t_end(ctx);
  CU(cudaGetLastError());
  size_t tmp = 0;
  CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp, ctx->b_seg_cnt.as<unsigned long long>(), ctx->b_seg_off.as<unsigned long long>(), (int)(ne + 1), ctx->stream));
  CU(ctx->b_cub.ensure(tmp));
  CU(cub::DeviceScan::ExclusiveSum(ctx->b_cub.p, tmp, ctx->b_seg_cnt.as<unsigned long long>(), ctx->b_seg_off.as<unsigned long long>(), (int)(ne + 1), ctx->stream));
  CU(cudaMemcpyAsync(&ctx->hd_scal[0], ctx->b_seg_off.as<unsigned long long>() + ne, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(&herr, derr, sizeof(Err), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  if (herr.block != ~0ull) {
    uint8_t code = 0;
    CU(cudaMemcpy(&code, ctx->b_blk_code.as<uint8_t>() + herr.block, 1, cudaMemcpyDeviceToHost));
    return fail(ctx, HM_ERR_ARG, REC_ERR[code == E_CRC ? E_CRC : E_INFLATE], pl->path ? pl->path : "", (long)herr.block);
  }
  if (herr.entry != ~0ull) return fail(ctx, HM_ERR_ARG, REC_ERR[E_BAI_ENTRY], pl->path ? pl->path : "", (long)herr.entry);
  const uint64_t n_rec = ctx->hd_scal[0];
  if (n_rec == 0) return HM_OK;
  if (n_rec >= (1ull << 31)) return fail(ctx, HM_ERR_ARG, "too many records in one region (%llu)", (unsigned long long)n_rec);
  CU(ctx->b_recoff.ensure(n_rec * 8));
  k_bam_walk<<<(unsigned)((ne + 127) / 128), 128, 0, ctx->stream>>>(buf, ctx->b_pentry.as<uint64_t>(), ne, pl->walk_end, nullptr,
                                                                     ctx->b_seg_off.as<unsigned long long>(), ctx->b_recoff.as<uint64_t>(), derr);
  CU(cudaGetLastError());
  // select and count
  const uint64_t stride = n_rec + 1;
  const int n_cnt = want_seq ? 5 : 4;
  CU(ctx->b_recinfo.ensure(n_rec * sizeof(RecInfo)));
  CU(ctx->b_cnt.ensure(n_cnt * stride * 8));
  CU(ctx->b_scan.ensure(n_cnt * stride * 8));
  CU(ctx->b_ecode.ensure(n_rec));
  CU(ctx->b_earg.ensure(n_rec * 8));
  t_begin(ctx, "k_bam_select");
  k_bam_select<<<(unsigned)((n_rec + 127) / 128), 128, 0, ctx->stream>>>(buf, ctx->b_recoff.as<uint64_t>(), n_rec, pl->walk_end, rid, start, end,
                                                                          ctx->b_recinfo.as<RecInfo>(), ctx->b_cnt.as<unsigned long long>(), n_cnt,
                                                                          ctx->b_ecode.as<uint8_t>(), ctx->b_earg.as<long long>(), derr);
  t_end(ctx);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(&herr, derr, sizeof(Err), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  const uint64_t stop = std::min<uint64_t>(herr.stop, n_rec);  // records from here on are never looked at by the host
  if (herr.rec < stop) return decode_record_error(ctx, pl, herr.rec);
  if (stop == 0) return HM_OK;
  // output offsets: exclusive scans of the counts (read index, first op, first quality byte, first name byte, and with
  // the base stream its first byte)
  unsigned long long* cnt = ctx->b_cnt.as<unsigned long long>();
  unsigned long long* scan = ctx->b_scan.as<unsigned long long>();
  tmp = 0;
  CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp, cnt, scan, (int)stride, ctx->stream));
  CU(ctx->b_cub.ensure(tmp));
  t_begin(ctx, "cub_scan_records");
  for (int k = 0; k < n_cnt; k++) CU(cub::DeviceScan::ExclusiveSum(ctx->b_cub.p, tmp, cnt + k * stride, scan + k * stride, (int)stride, ctx->stream));
  t_end(ctx);
  for (int k = 0; k < n_cnt; k++) CU(cudaMemcpyAsync(&ctx->hd_scal[k], scan + k * stride + stop, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  const uint64_t n = ctx->hd_scal[0], n_ops = ctx->hd_scal[1], n_bq = ctx->hd_scal[2], n_nm = ctx->hd_scal[3];
  const uint64_t n_seq = want_seq ? ctx->hd_scal[4] : 0;
  // the resident batch's buffers, written in place
  CU(ctx->b_tstart.ensure(n * 4 + 16)); CU(ctx->b_tend.ensure(n * 4 + 16)); CU(ctx->b_qstart.ensure(n * 4 + 16));
  CU(ctx->b_qlen.ensure(n * 4 + 16)); CU(ctx->b_mapq.ensure(n + 16)); CU(ctx->b_flags.ensure(n + 16)); CU(ctx->b_qname.ensure(n * 4 + 16));
  CU(ctx->b_n_ops.ensure(n * 4 + 16)); CU(ctx->b_bq_off.ensure(n * 8 + 16)); CU(ctx->b_op_off.ensure(n * 8 + 16));
  CU(ctx->b_bq.ensure(n_bq + 32)); CU(ctx->b_ops.ensure(n_ops * 4 + 16)); CU(ctx->b_names.ensure(n_nm + 16));
  CU(ctx->b_name_off.ensure(n * 8 + 16));
  if (want_seq) { CU(ctx->b_seq.ensure(n_seq + 32)); CU(ctx->b_seq_off.ensure(n * 8 + 16)); }
  ParseOut o{ctx->b_tstart.as<int32_t>(), ctx->b_tend.as<int32_t>(), ctx->b_qstart.as<int32_t>(), ctx->b_qlen.as<int32_t>(),
             ctx->b_mapq.as<uint8_t>(), ctx->b_flags.as<uint8_t>(), ctx->b_n_ops.as<uint32_t>(), ctx->b_bq_off.as<uint64_t>(),
             ctx->b_op_off.as<uint64_t>(), ctx->b_name_off.as<uint64_t>(), ctx->b_bq.as<uint8_t>(), ctx->b_ops.as<uint32_t>(),
             ctx->b_names.as<char>(), want_seq ? ctx->b_seq_off.as<uint64_t>() : nullptr, want_seq ? ctx->b_seq.as<uint8_t>() : nullptr};
  t_begin(ctx, "k_bam_parse");
  k_bam_parse<<<(unsigned)((stop * 32 + 255) / 256), 256, 0, ctx->stream>>>(buf, ctx->b_recinfo.as<RecInfo>(), stop, scan, stride, o,
                                                                             ctx->b_ecode.as<uint8_t>(), ctx->b_earg.as<long long>(), derr);
  t_end(ctx);
  CU(cudaGetLastError());
  if (!ctx->hd_tstart.resize(n) || !ctx->hd_tend.resize(n) || !ctx->hd_qstart.resize(n) || !ctx->hd_qlen.resize(n) ||
      !ctx->hd_n_ops.resize(n) || !ctx->hd_bq_off.resize(n) || !ctx->hd_op_off.resize(n) || !ctx->hd_name_off.resize(n) ||
      !ctx->hd_names.resize(n_nm + 1) || (want_seq && !ctx->hd_seq_off.resize(n)))
    return fail(ctx, HM_ERR_ARG, "out of page-locked host memory for %llu reads", (unsigned long long)n);
  t_begin(ctx, "d2h_reads_names");
#define DOWN(h, d, bytes) CU(cudaMemcpyAsync(ctx->h.data(), ctx->d.p, (bytes), cudaMemcpyDeviceToHost, ctx->stream))
  DOWN(hd_tstart, b_tstart, n * 4); DOWN(hd_tend, b_tend, n * 4); DOWN(hd_qstart, b_qstart, n * 4); DOWN(hd_qlen, b_qlen, n * 4);
  DOWN(hd_n_ops, b_n_ops, n * 4); DOWN(hd_bq_off, b_bq_off, n * 8); DOWN(hd_op_off, b_op_off, n * 8);
  DOWN(hd_name_off, b_name_off, n * 8); DOWN(hd_names, b_names, n_nm);
  if (want_seq) DOWN(hd_seq_off, b_seq_off, n * 8);
#undef DOWN
  t_end(ctx);
  CU(cudaMemcpyAsync(&herr, derr, sizeof(Err), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  if (herr.parse != ~0ull) return decode_record_error(ctx, pl, herr.parse);
  ctx->dec_n = n;
  ctx->dec_ops = n_ops;
  ctx->dec_bq = n_bq ? n_bq : 16;
  if (want_seq) ctx->dec_seq = n_seq ? n_seq : 16;
  *n_reads = n;
  return HM_OK;
}

// stage: 0 the whole call, 1 enqueue only (hm_call_chunks_submit), 2 everything after the enqueue (hm_call_chunks_collect)
static int call_chunks_impl(hm_ctx* ctx, const hm_chunk* chunks, size_t n_chunks, hm_site_record* out, size_t cap, size_t* n_out,
                           int64_t log[HM_CALL_LOG_LEN], bool async, int stage = 0);

int hm_call_chunks(hm_ctx* ctx, const hm_chunk* chunks, size_t n_chunks, hm_site_record* out, size_t cap, size_t* n_out,
                   int64_t log[HM_CALL_LOG_LEN]) {
  return call_chunks_impl(ctx, chunks, n_chunks, out, cap, n_out, log, false);
}

/* hm_call_chunks in two halves, so that a host that drives several contexts (the chunk runs of a genome on one GPU) keeps
 * the device busy: submit enqueues the whole device path of the call and returns at once; collect waits for it and
 * does what hm_call_chunks_async does after its synchronisation (counters, som_seen replay, record copy).  One call
 * may be pending per context; nothing else may be asked of the context in between. */
int hm_call_chunks_submit(hm_ctx* ctx, const hm_chunk* chunks, size_t n_chunks) {
  if (ctx && ctx->pend.active) return fail(ctx, HM_ERR_STATE, "a submitted call is still pending: collect it first");
  size_t n_out = 0;
  int64_t log[HM_CALL_LOG_LEN];
  return call_chunks_impl(ctx, chunks, n_chunks, nullptr, 0, &n_out, log, true, 1);
}
int hm_call_chunks_collect(hm_ctx* ctx, hm_site_record* out, size_t cap, size_t* n_out, int64_t log[HM_CALL_LOG_LEN]) {
  if (!ctx) return HM_ERR_ARG;
  if (!ctx->pend.active) return fail(ctx, HM_ERR_STATE, "no submitted call is pending");
  ctx->pend.active = false;
  return call_chunks_impl(ctx, ctx->pend.chunks.data(), ctx->pend.chunks.size(), out, cap, n_out, log, true, 2);
}

/* hm_call_chunks that returns as soon as the counters are final: the record copy into `out` may still be in
 * flight (on the context's copy stream) and overlaps whatever the caller enqueues next; hm_records_wait blocks
 * until `out` is complete.  Two calls may be in flight: `out` must not be reused before the second next call. */
int hm_call_chunks_async(hm_ctx* ctx, const hm_chunk* chunks, size_t n_chunks, hm_site_record* out, size_t cap, size_t* n_out,
                         int64_t log[HM_CALL_LOG_LEN]) {
  return call_chunks_impl(ctx, chunks, n_chunks, out, cap, n_out, log, true);
}

int hm_set_option(hm_ctx* ctx, int option, int value) {
  if (!ctx) return HM_ERR_ARG;
  if (option == HM_OPT_OMIT_RESTATEMENTS) { ctx->omit_restatements = value != 0; return HM_OK; }
  if (option == HM_OPT_KERNEL_TIMING) { ctx->ktiming = value != 0; return HM_OK; }
  return fail(ctx, HM_ERR_ARG, "unknown option %d", option);
}

int hm_records_wait(hm_ctx* ctx) {
  if (!ctx) return HM_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  int rc = flush_deferred(ctx, false);
  if (rc) return rc;
  if (ctx->copy_pending) { CU(cudaStreamSynchronize(ctx->copy_stream)); ctx->copy_pending = false; }
  return HM_OK;
}

// ---- the fused path (callfused.cuh): everything between the uploads and the one synchronisation of a call ----
namespace {

inline size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }

// can the fused path run this call?  (else the first version does: chunk spans of 2^27 positions and more, more than
// 2^32 (chunk, read) pairs or candidate slots — nothing a reference-style chunk list produces)
bool fused_eligible(hm_ctx* ctx, const hm_chunk* chunks, size_t n_chunks, uint64_t n_pairs, uint64_t* total_cap, uint64_t* n_tiles) {
  const bool force_v1 = getenv("HIMUT_B200_CALL_V1") != nullptr; // read per call: tests switch it
  if (force_v1 || n_pairs == 0 || n_pairs >= 0xffffffffull) return false;
  uint64_t cap = 0, tiles = 0;
  for (size_t i = 0; i < n_chunks; i++) {
    const int64_t span = (int64_t)chunks[i].end - (int64_t)chunks[i].start;
    if (span >= (1ll << HC_KEY_POS_BITS)) return false;
    cap += ctx->h_ops_prefix[chunks[i].read_hi] - ctx->h_ops_prefix[chunks[i].read_lo];
    if (span >= 0) tiles += (uint64_t)(span >> HC_TILE_BITS) + 1;
  }
  if (cap >= 0xffffffffull || tiles >= (1ull << 31)) return false;
  *total_cap = cap; *n_tiles = tiles;
  return true;
}

struct FusedGeom { // device pointers into the one geometry block of a call
  const hm_chunk* chunks; const uint64_t* pair_off; const uint64_t* seg_off; const uint32_t* tile_off; const int32_t* geom;
  const uint32_t* tile_chunk;
};

// enqueue the fused path on ctx->stream.  *site_cap: distinct sites the buffers hold (k_tile_scan flags an overflow).
int fused_enqueue(hm_ctx* ctx, const hm_chunk* chunks, size_t n_chunks, const std::vector<uint64_t>& pair_off, const int32_t* geom,
                  uint64_t total_cap, uint64_t n_tiles, uint64_t site_cap, int parity, bool omit, size_t boundary_cap, FusedGeom* G_out) {
  const uint64_t n_pairs = pair_off.back();
  // ---- geometry: one pinned block, one copy ----
  const size_t o_chunks = 0, o_pair = align16(o_chunks + n_chunks * sizeof(hm_chunk)), o_seg = align16(o_pair + (n_chunks + 1) * 8),
               o_tile = align16(o_seg + (n_chunks + 1) * 8), o_geom = align16(o_tile + (n_chunks + 1) * 4),
               o_tchunk = align16(o_geom + 2 * n_chunks * 4 + 16), g_bytes = align16(o_tchunk + (size_t)n_tiles * 4 + 16);
  if (g_bytes > ctx->h_geom_cap) {
    if (ctx->h_geom_pin) cudaFreeHost(ctx->h_geom_pin);
    ctx->h_geom_pin = nullptr; ctx->h_geom_cap = 0;
    CU(cudaHostAlloc((void**)&ctx->h_geom_pin, g_bytes + g_bytes / 4, cudaHostAllocMapped));
    ctx->h_geom_cap = g_bytes + g_bytes / 4;
  }
  char* hp = ctx->h_geom_pin;
  memcpy(hp + o_chunks, chunks, n_chunks * sizeof(hm_chunk));
  memcpy(hp + o_pair, pair_off.data(), (n_chunks + 1) * 8);
  uint64_t* h_seg = reinterpret_cast<uint64_t*>(hp + o_seg);
  uint32_t* h_tile = reinterpret_cast<uint32_t*>(hp + o_tile);
  uint32_t* h_tchunk = reinterpret_cast<uint32_t*>(hp + o_tchunk);
  h_seg[0] = 0; h_tile[0] = 0;
  for (size_t i = 0; i < n_chunks; i++) {
    const int64_t span = (int64_t)chunks[i].end - (int64_t)chunks[i].start;
    const uint32_t nt = span >= 0 ? (uint32_t)(span >> HC_TILE_BITS) + 1u : 0u;
    h_seg[i + 1] = h_seg[i] + (ctx->h_ops_prefix[chunks[i].read_hi] - ctx->h_ops_prefix[chunks[i].read_lo]);
    for (uint32_t k = 0; k < nt; k++) h_tchunk[h_tile[i] + k] = (uint32_t)i;
    h_tile[i + 1] = h_tile[i] + nt;
  }
  memcpy(hp + o_geom, geom, 2 * n_chunks * 4);
  CU(ctx->b_cgeom.ensure(g_bytes));
  { // g_bytes is a multiple of 16
    void* mapped = nullptr;
    CU(cudaHostGetDevicePointer(&mapped, hp, 0));
    const uint32_t n16 = (uint32_t)(g_bytes / 16);
    k_fetch_block<<<std::max(1u, std::min(32u, (n16 + 255u) / 256u)), 256, 0, ctx->stream>>>(reinterpret_cast<const uint4*>(mapped), ctx->b_cgeom.as<uint4>(), n16);
    CU(cudaGetLastError());
  }
  char* dp = ctx->b_cgeom.as<char>();
  FusedGeom G = {reinterpret_cast<const hm_chunk*>(dp + o_chunks), reinterpret_cast<const uint64_t*>(dp + o_pair),
                 reinterpret_cast<const uint64_t*>(dp + o_seg), reinterpret_cast<const uint32_t*>(dp + o_tile),
                 reinterpret_cast<const int32_t*>(dp + o_geom), reinterpret_cast<const uint32_t*>(dp + o_tchunk)};
  *G_out = G;

  // ---- buffers ----
  const size_t capk = (size_t)std::max<uint64_t>(total_cap, 1);
  CU(ctx->b_seg_keys.ensure(capk * 4 + 16)); CU(ctx->b_seg_read.ensure(capk * 4 + 16));
  CU(ctx->b_keys_tmp.ensure(capk * 4 + 16)); CU(ctx->b_gscratch.ensure(capk * 8 + 16));
  const size_t z_cnt = 0, z_cur = z_cnt + n_chunks * 4, z_cur2 = z_cur + n_chunks * 4, z_bytes = align16(z_cur2 + n_chunks * 4) + 16;
  CU(ctx->b_czero.ensure(z_bytes));
  CU(ctx->b_pair_c.ensure((size_t)n_pairs * 4 + 16));
  CU(ctx->b_tiles.ensure(((size_t)n_tiles * 3 + 4) * 4));
  const uint64_t stride = (site_cap + 31) & ~31ull;
  const uint32_t n_slots = ctx->site_slots;
  if (stride * n_slots + site_cap >= (1ull << 32)) return fail(ctx, HM_ERR_ARG, "%llu candidate sites in one call: split the chunk list", (unsigned long long)site_cap);
  CU(ctx->b_keys.ensure(site_cap * 8 + 16));
  CU(ctx->b_agg.ensure(stride * n_slots * 4 + site_cap * 8 + 16));
  CU(ctx->b_compact[parity].ensure(site_cap * sizeof(hm_site_record)));
  const unsigned n_red = (unsigned)((site_cap + 127) / 128);
  CU(ctx->b_bidx.ensure(boundary_cap * 4 + HM_BOUNDARY_FIRST * 4));
  CU(ctx->b_brecs.ensure((boundary_cap + HM_BOUNDARY_FIRST) * sizeof(hm_site_record)));
  CU(ctx->b_bpos.ensure((boundary_cap + HM_BOUNDARY_FIRST) * 4));
  const size_t qseen_bytes = ((size_t)ctx->max_qname_id + 4) & ~(size_t)3; // one byte per query name, set through 32-bit atomics
  CU(ctx->b_qseen.ensure(qseen_bytes + 16));
  if (ctx->params.phase) CU(ctx->b_pair_hap.ensure(n_pairs + 16));

  char* z = ctx->b_czero.as<char>();
  uint32_t* seg_cnt = reinterpret_cast<uint32_t*>(z + z_cnt);
  uint32_t* cursor = reinterpret_cast<uint32_t*>(z + z_cur);
  uint32_t* cursor2 = reinterpret_cast<uint32_t*>(z + z_cur2);
  uint32_t* tile_src = ctx->b_tiles.as<uint32_t>();
  uint32_t* tile_cnt = tile_src + n_tiles;
  uint32_t* tile_dst = tile_cnt + n_tiles; // n_tiles + 1 entries
  unsigned long long* d_cnt = ctx->b_counters.as<unsigned long long>();
  unsigned long long* keys = ctx->b_keys.as<unsigned long long>();
  uint32_t* entries = ctx->b_agg.as<uint32_t>();
  uint32_t* site_lo = entries + stride * n_slots;
  uint32_t* site_n = site_lo + site_cap;
  uint8_t* pair_hap = ctx->params.phase ? ctx->b_pair_hap.as<uint8_t>() : nullptr;
  uint32_t* pair_c = ctx->b_pair_c.as<uint32_t>();
  const bool has_seq = ctx->db.seq != nullptr;

  static bool attr_set = false;
  const size_t sort_smem = (2 * (size_t)HC_TILE_WORDS + 2 * (size_t)HC_CAPD + (size_t)HC_STAGE) * 4;
  const size_t scan_smem = sizeof(ScanWarp) * HC_SCAN_WARPS;
  const size_t pairs_smem = (size_t)HC_A_CAP * 4;
  if (!attr_set) {
    CU(cudaFuncSetAttribute(k_site_sort, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sort_smem));
    CU(cudaFuncSetAttribute(k_call_pairs<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pairs_smem));
    CU(cudaFuncSetAttribute(k_call_pairs<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pairs_smem));
    CU(cudaFuncSetAttribute(k_call_scan<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)scan_smem));
    CU(cudaFuncSetAttribute(k_call_scan<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)scan_smem));
    attr_set = true;
  }

  CU(cudaMemsetAsync(ctx->b_counters.p, 0, 256, ctx->stream));
  CU(cudaMemsetAsync(ctx->b_qseen.p, 0, qseen_bytes, ctx->stream));
  CU(cudaMemsetAsync(ctx->b_czero.p, 0, z_bytes, ctx->stream));
  const unsigned pair_blocks_a = (unsigned)((n_pairs + 127) / 128);
  t_begin(ctx, "k_call_pairs");
  if (has_seq)
    k_call_pairs<true><<<pair_blocks_a, 128, pairs_smem, ctx->stream>>>(ctx->db, ctx->dp, ctx->dphase, G.chunks, (uint32_t)n_chunks, G.pair_off, n_pairs, pair_c, pair_hap,
                                                              ctx->b_qseen.as<uint32_t>(), d_cnt + 24, G.seg_off, seg_cnt,
                                                              ctx->b_seg_keys.as<uint32_t>(), ctx->b_seg_read.as<uint32_t>());
  else
    k_call_pairs<false><<<pair_blocks_a, 128, pairs_smem, ctx->stream>>>(ctx->db, ctx->dp, ctx->dphase, G.chunks, (uint32_t)n_chunks, G.pair_off, n_pairs, pair_c, pair_hap,
                                                               ctx->b_qseen.as<uint32_t>(), d_cnt + 24, G.seg_off, seg_cnt,
                                                               ctx->b_seg_keys.as<uint32_t>(), ctx->b_seg_read.as<uint32_t>());
  t_end(ctx);
  CU(cudaGetLastError());
  t_begin(ctx, "k_site_sort");
  if (n_tiles)
    k_site_sort<<<(unsigned)n_tiles, HC_SORT_THREADS, sort_smem, ctx->stream>>>(G.tile_chunk, G.tile_off, G.seg_off, seg_cnt, ctx->b_seg_keys.as<uint32_t>(),
                                                                               cursor, cursor2, ctx->b_gscratch.as<uint32_t>(), ctx->b_keys_tmp.as<uint32_t>(),
                                                                               tile_src, tile_cnt);
  k_tile_scan<<<1, 1024, 0, ctx->stream>>>(tile_cnt, (uint32_t)n_tiles, tile_dst, (unsigned long long)site_cap, d_cnt);
  k_site_range2<<<(unsigned)((site_cap + 255) / 256), 256, 0, ctx->stream>>>(ctx->db, G.chunks, G.tile_chunk, tile_src, tile_dst, (uint32_t)n_tiles,
                                                                            ctx->b_keys_tmp.as<uint32_t>(), d_cnt + 1, keys, site_lo, site_n, entries, stride, n_slots);
  t_end(ctx);
  CU(cudaGetLastError());
  int rc = flush_deferred(ctx, true); // the previous call's records start moving now, under k_call_scan
  if (rc) return rc;
  const unsigned pair_blocks_b = (unsigned)((n_pairs + HC_SCAN_WARPS - 1) / HC_SCAN_WARPS);
  t_begin(ctx, "k_call_scan");
  if (has_seq)
    k_call_scan<true><<<pair_blocks_b, 32 * HC_SCAN_WARPS, scan_smem, ctx->stream>>>(ctx->db, ctx->dp, G.chunks, G.pair_off, n_pairs, pair_c, pair_hap,
                                                                                    G.tile_off, tile_dst, keys, site_lo, site_n, entries, (uint32_t)stride,
                                                                                    d_cnt + 1, n_slots);
  else
    k_call_scan<false><<<pair_blocks_b, 32 * HC_SCAN_WARPS, scan_smem, ctx->stream>>>(ctx->db, ctx->dp, G.chunks, G.pair_off, n_pairs, pair_c, pair_hap,
                                                                                     G.tile_off, tile_dst, keys, site_lo, site_n, entries, (uint32_t)stride,
                                                                                     d_cnt + 1, n_slots);
  t_end(ctx);
  CU(cudaGetLastError());
  CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_copy_done[parity], 0)); // the copy that last read this record buffer
  t_begin(ctx, "k_site_reduce");
  k_site_reduce<<<n_red, 128, 0, ctx->stream>>>(ctx->db, ctx->dp, ctx->dsets, ctx->dlut, ctx->dphase, ctx->dup_names ? 1 : 0, G.chunks, G.pair_off, pair_hap,
                                                G.geom, G.geom + n_chunks, keys, d_cnt + 1, site_lo, site_n, entries, stride,
                                                nullptr, d_cnt + 8, ctx->b_bidx.as<uint32_t>(), ctx->b_brecs.as<hm_site_record>(),
                                                (uint32_t)boundary_cap, d_cnt + 4, reinterpret_cast<int*>(d_cnt + 3),
                                                ctx->b_compact[parity].as<hm_site_record>(), d_cnt + 6, ctx->b_bpos.as<uint32_t>(), omit ? 1 : 0, n_slots);
  t_end(ctx);
  CU(cudaGetLastError());
  return HM_OK;
}

}  // namespace

static int call_chunks_impl(hm_ctx* ctx, const hm_chunk* chunks, size_t n_chunks, hm_site_record* out, size_t cap, size_t* n_out,
                            int64_t log[HM_CALL_LOG_LEN], bool async, int stage) {
  int rc = check_ready(ctx, chunks, n_chunks);
  if (rc) return rc;
  if (stage != 2 && ctx->pend.active) return fail(ctx, HM_ERR_STATE, "a submitted call is still pending: collect it first");
  if (!log || !n_out) return fail(ctx, HM_ERR_ARG, "log / n_out is NULL");
  CU(cudaSetDevice(ctx->device));
  // HIMUT_B200_HOST_TIMING=1: wall-clock of the host-visible phases of one call, to stderr (diagnostics)
  static const bool host_timing = getenv("HIMUT_B200_HOST_TIMING") != nullptr;
  auto tp0 = std::chrono::steady_clock::now();
  double ht[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  auto lap = [&](int i) { auto t = std::chrono::steady_clock::now(); ht[i] += std::chrono::duration<double, std::milli>(t - tp0).count(); tp0 = t; };
  memset(log, 0, sizeof(int64_t) * HM_CALL_LOG_LEN);
  *n_out = 0;
  ctx->final_recs.clear();
  if (stage != 2) t_reset(ctx);
  std::vector<uint64_t> pair_off(n_chunks + 1, 0);
  for (size_t i = 0; i < n_chunks; i++) pair_off[i + 1] = pair_off[i] + (chunks[i].read_hi - chunks[i].read_lo);
  const uint64_t n_pairs = pair_off.back();
  uint64_t total_cap = 0, n_tiles = 0;
  const bool fused = fused_eligible(ctx, chunks, n_chunks, n_pairs, &total_cap, &n_tiles);
  ctx->call_path = fused ? 2 : 1;
  ctx->own_launch_count = false;
  if (!fused) {
    if ((rc = upload(ctx, ctx->b_chunks, chunks, n_chunks))) return rc;
    if ((rc = upload(ctx, ctx->b_pair_off, pair_off.data(), pair_off.size()))) return rc;
  }
  // chunk geometry for the som_seen carry: a position can only have been claimed by an earlier
  // chunk if it lies at or below the largest chunk end seen so far, and only needs remembering if
  // a later chunk starts at or below it.  With the reference's own chunking that is just the
  // shared boundary position, so very few records ever reach the host replay.
  std::vector<int32_t> geom(2 * n_chunks + 2);
  int32_t* prev_max_end = geom.data();
  int32_t* next_min_start = geom.data() + n_chunks;
  {
    int32_t m = INT32_MIN;
    for (size_t i = 0; i < n_chunks; i++) { prev_max_end[i] = m; m = std::max(m, chunks[i].end); }
    m = INT32_MAX;
    for (size_t i = n_chunks; i-- > 0;) { next_min_start[i] = m; m = std::min(m, chunks[i].start); }
  }

  // counters (u64): [0] n_keys (first version), [1] n_unique, [2] num_ccs, [3] error flag, [4] n_boundary,
  // [5] sites needed when the fused path's site buffers overflowed, [6] records kept by k_compact_sites,
  // [8..23] status histogram, [24..31] num_ccs of the fused path in eight slots
  const size_t CNT_BYTES = 256;
  CU(ctx->b_counters.ensure(CNT_BYTES));
  if (!ctx->h_cnt_pin) CU(cudaHostAlloc((void**)&ctx->h_cnt_pin, CNT_BYTES + HM_BOUNDARY_FIRST * (8 + sizeof(hm_site_record)), cudaHostAllocMapped));
  unsigned long long h_cnt[32];
  memset(h_cnt, 0, sizeof(h_cnt));
  unsigned long long* d_cnt = ctx->b_counters.as<unsigned long long>();
  const int parity = stage == 2 ? ctx->pend.parity : ctx->rec_parity;
  DevBuf& rec_buf = parity ? ctx->b_records_alt : ctx->b_records;
  const bool omit = stage == 2 ? ctx->pend.omit : ctx->omit_restatements;
  size_t HM_BOUNDARY_CAP = HM_BOUNDARY_CAP_DEFAULT;
  if (const char* e = getenv("HIMUT_B200_BOUNDARY_CAP")) HM_BOUNDARY_CAP = (size_t)std::max(0ll, atoll(e));
  if (stage == 1 && !fused) { // the first version synchronises in the middle: everything happens at collect
    ctx->pend.active = true;
    ctx->pend.chunks.assign(chunks, chunks + n_chunks);
    ctx->pend.parity = parity; ctx->pend.omit = omit;
    return HM_OK;
  }
  uint32_t* h_bidx = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(ctx->h_cnt_pin) + CNT_BYTES);
  uint32_t* h_bpos = h_bidx + HM_BOUNDARY_FIRST;
  hm_site_record* h_brecs = reinterpret_cast<hm_site_record*>(h_bpos + HM_BOUNDARY_FIRST);
  unsigned long long n_keys = 0;

  if (fused) {
    uint64_t site_cap = std::max<uint64_t>(std::max<uint64_t>(ctx->site_cap_hint, ctx->n_ops_total / 8), 4096);
    if (const char* e = getenv("HIMUT_B200_SITE_CAP")) site_cap = (uint64_t)std::max(1ll, atoll(e)); // tests: force the overflow retry
    site_cap = std::min<uint64_t>(site_cap, std::max<uint64_t>(total_cap, 1));
    size_t bcap = HM_BOUNDARY_CAP;
    int n_launched = 0;
    if (stage == 2) { site_cap = ctx->pend.site_cap; bcap = ctx->pend.bcap; n_launched = ctx->pend.n_launched; }
    for (int attempt = 0;; attempt++) {
      if (!(stage == 2 && attempt == 0)) { // collect: the first attempt was enqueued by submit
        t_reset(ctx);
        FusedGeom G;
        if ((rc = fused_enqueue(ctx, chunks, n_chunks, pair_off, geom.data(), total_cap, n_tiles, site_cap, parity, omit, bcap, &G))) return rc;
        k_publish_call<<<8, 256, 0, ctx->stream>>>(reinterpret_cast<const uint32_t*>(d_cnt), (uint32_t)(CNT_BYTES / 4), ctx->b_bidx.as<uint32_t>(),
                                                   ctx->b_bpos.as<uint32_t>(), ctx->b_brecs.as<uint32_t>(), (uint32_t)std::min<size_t>(HM_BOUNDARY_FIRST, bcap),
                                                   d_cnt + 4, reinterpret_cast<uint32_t*>(ctx->h_cnt_pin), h_bidx, h_bpos, reinterpret_cast<uint32_t*>(h_brecs));
        CU(cudaGetLastError());
        // own kernels launched by this attempt: k_fetch_block, k_call_pairs, k_site_sort, k_tile_scan, k_site_range2, k_call_scan,
        // k_site_reduce, k_publish_call (+ k_bq_expand / k_bq_sum, counted by the upload)
        n_launched += 7 + (n_tiles ? 1 : 0);
      }
      if (stage == 1) { // submitted: the rest happens at collect
        ctx->pend.active = true;
        ctx->pend.chunks.assign(chunks, chunks + n_chunks);
        ctx->pend.site_cap = site_cap; ctx->pend.bcap = bcap; ctx->pend.n_launched = n_launched;
        ctx->pend.parity = parity; ctx->pend.omit = omit;
        return HM_OK;
      }
      lap(4);
      CU(cudaStreamSynchronize(ctx->stream)); // the one synchronisation of the call
      lap(5);
      memcpy(h_cnt, ctx->h_cnt_pin, CNT_BYTES);
      const bool more_sites = h_cnt[5] != 0, more_boundary = h_cnt[4] > bcap;
      if (!more_sites && !more_boundary) break;
      if (attempt >= 3) return fail(ctx, HM_ERR_STATE, "site / boundary buffers overflowed repeatedly (%llu sites, %llu boundary records)", h_cnt[5], h_cnt[4]);
      // a list overflowed: run again with room (the counts are exact now)
      if (more_sites) site_cap = std::min<uint64_t>(h_cnt[5] + h_cnt[5] / 8 + 1024, std::max<uint64_t>(total_cap, 1));
      if (more_boundary) bcap = (size_t)h_cnt[4] + 1024;
      memset(h_cnt, 0, sizeof(h_cnt));
    }
    HM_BOUNDARY_CAP = bcap;
    ctx->own_launch_count = true;
    ctx->last_launches = n_launched;
    h_cnt[2] = 0;
    for (int k = 24; k < 32; k++) h_cnt[2] += h_cnt[k]; // num_ccs: distinct query names, counted in eight slots
    ctx->site_cap_hint = std::max<uint64_t>(ctx->site_cap_hint, h_cnt[1] + h_cnt[1] / 4);
    n_keys = h_cnt[1];
  } else {
  if (n_chunks && (rc = upload(ctx, ctx->b_geom, geom.data(), 2 * n_chunks))) return rc;
  if ((rc = launch_read_scan(ctx))) return rc;
  CU(ctx->b_qseen.ensure((size_t)ctx->max_qname_id + 1));
  if (ctx->params.phase) CU(ctx->b_pair_hap.ensure(n_pairs + 16));
  unsigned long long key_cap = std::max<unsigned long long>(ctx->n_ops_total, 1024);
  // bits of (tpos - chunk.start): candidates satisfy start <= tpos <= end (is_chunk, caller.py:325)
  int pos_bits = 1;
  for (size_t i = 0; i < n_chunks; i++) {
    const int64_t span = (int64_t)chunks[i].end - (int64_t)chunks[i].start;
    while (pos_bits < 32 && span >= (1ll << pos_bits)) pos_bits++;
  }
  int end_bit = pos_bits + 4;
  for (size_t c = n_chunks; c > 0; c >>= 1) end_bit++;
  end_bit = std::min(end_bit, 64);
  for (int attempt = 0; attempt < 2 && n_pairs; attempt++) {
    CU(ctx->b_keys.ensure(key_cap * 8));
    { // everything the sort needs that does not depend on the candidate count: done while the device works
      CU(ctx->b_keys_sorted.ensure(key_cap * 8));
      size_t tmp_sort = 0, tmp_uniq = 0;
      unsigned long long* k_in = ctx->b_keys.as<unsigned long long>();
      unsigned long long* k_sorted = ctx->b_keys_sorted.as<unsigned long long>();
      CU(cub::DeviceRadixSort::SortKeys(nullptr, tmp_sort, k_in, k_sorted, (int64_t)key_cap, 0, end_bit, ctx->stream));
      CU(cub::DeviceSelect::Unique(nullptr, tmp_uniq, k_sorted, k_in, ctx->b_counters.as<unsigned long long>() + 1, (int64_t)key_cap, ctx->stream));
      CU(ctx->b_cub.ensure(std::max(tmp_sort, tmp_uniq)));
    }
    CU(cudaMemsetAsync(ctx->b_counters.p, 0, CNT_BYTES, ctx->stream));
    CU(cudaMemsetAsync(ctx->b_qseen.p, 0, (size_t)ctx->max_qname_id + 1, ctx->stream));
    const unsigned blocks = (unsigned)((n_pairs * 32 + 255) / 256);
    t_begin(ctx, "k_candidates");
    k_candidates<<<blocks, 256, 0, ctx->stream>>>(ctx->db, ctx->dp, ctx->dphase, ctx->b_chunks.as<hm_chunk>(), (uint32_t)n_chunks,
                                                  ctx->b_pair_off.as<uint64_t>(), n_pairs,
                                                  ctx->params.phase ? ctx->b_pair_hap.as<uint8_t>() : nullptr,
                                                  ctx->b_qseen.as<uint8_t>(), ctx->b_keys.as<unsigned long long>(), key_cap, d_cnt, pos_bits);
    t_end(ctx);
    CU(cudaGetLastError());
    lap(0); // uploads + launches up to k_candidates
    k_publish<<<1, 32, 0, ctx->stream>>>(reinterpret_cast<const uint32_t*>(d_cnt), reinterpret_cast<uint32_t*>(ctx->h_cnt_pin), 2);
    CU(cudaStreamSynchronize(ctx->stream));
    h_cnt[0] = ctx->h_cnt_pin[0];
    lap(1); // sync 1: candidate count
    if (h_cnt[0] <= key_cap) break;
    key_cap = h_cnt[0];
  }
  n_keys = h_cnt[0];

  if (n_pairs) {
    if (n_keys) {
      // sort + unique of the candidate keys (library plumbing: cub), then the site kernels
      size_t tmp_sort = ctx->b_cub.cap, tmp_uniq = ctx->b_cub.cap; // sized for key_cap >= n_keys above
      unsigned long long* k_in = ctx->b_keys.as<unsigned long long>();
      unsigned long long* k_sorted = ctx->b_keys_sorted.as<unsigned long long>();
      t_begin(ctx, "cub_sort_unique_keys");
      CU(cub::DeviceRadixSort::SortKeys(ctx->b_cub.p, tmp_sort, k_in, k_sorted, (int64_t)n_keys, 0, end_bit, ctx->stream));
      CU(cub::DeviceSelect::Unique(ctx->b_cub.p, tmp_uniq, k_sorted, k_in, d_cnt + 1, (int64_t)n_keys, ctx->stream));
      k_expand_keys<<<(unsigned)((n_keys + 255) / 256), 256, 0, ctx->stream>>>(k_in, d_cnt + 1, ctx->b_chunks.as<hm_chunk>(), pos_bits);
      t_end(ctx);
      if ((rc = flush_deferred(ctx, true))) return rc; // the previous call's records start moving behind the sort
      k_publish<<<1, 32, 0, ctx->stream>>>(reinterpret_cast<const uint32_t*>(d_cnt + 1), reinterpret_cast<uint32_t*>(ctx->h_cnt_pin + 1), 2);
      lap(2); // sort / unique launches
      CU(cudaStreamSynchronize(ctx->stream));
      h_cnt[1] = ctx->h_cnt_pin[1];
      lap(3); // sync 2: distinct count
      const size_t n_unique = (size_t)h_cnt[1];
      const uint64_t stride = (n_unique + 31) & ~31ull;
      CU(ctx->b_agg.ensure(stride * HM_SITE_SLOTS * 4 + n_unique * 8));
      uint32_t* entries = ctx->b_agg.as<uint32_t>();
      uint32_t* site_lo = entries + stride * HM_SITE_SLOTS;
      uint32_t* site_n = site_lo + n_unique;
      CU(rec_buf.ensure(n_unique * sizeof(hm_site_record)));
      CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_copy_done[parity], 0)); // the copy that last read this buffer
      CU(ctx->b_bidx.ensure((size_t)HM_BOUNDARY_CAP * 4 + HM_BOUNDARY_FIRST * 4));
      CU(ctx->b_brecs.ensure(((size_t)HM_BOUNDARY_CAP + HM_BOUNDARY_FIRST) * sizeof(hm_site_record)));
      t_begin(ctx, "k_site_range");
      k_site_range<<<(unsigned)((n_unique + 255) / 256), 256, 0, ctx->stream>>>(ctx->db, ctx->b_chunks.as<hm_chunk>(), k_in, d_cnt + 1,
                                                                              site_lo, site_n);
      t_end(ctx);
      CU(cudaGetLastError());
      CU(ctx->b_koff.ensure((n_chunks + 2) * 4));
      t_begin(ctx, "k_site_entries_by_read");
      CU(cudaMemsetAsync(entries, 0xff, stride * HM_SITE_SLOTS * 4, ctx->stream));
      k_chunk_key_ranges<<<(unsigned)((n_chunks + 1 + 127) / 128), 128, 0, ctx->stream>>>(k_in, d_cnt + 1, (uint32_t)n_chunks, ctx->b_koff.as<uint32_t>());
      auto gather = ctx->db.seq ? k_site_entries_by_read<true> : k_site_entries_by_read<false>;
      gather<<<(unsigned)((n_pairs * 32 + 255) / 256), 256, 0, ctx->stream>>>(
          ctx->db, ctx->dp, ctx->b_chunks.as<hm_chunk>(), (uint32_t)n_chunks, ctx->b_pair_off.as<uint64_t>(), n_pairs,
          ctx->b_pair_hap.as<uint8_t>(), k_in, ctx->b_koff.as<uint32_t>(), site_lo, site_n, entries, stride);
      t_end(ctx);
      CU(cudaGetLastError());
      t_begin(ctx, "k_site_reduce");
      k_site_reduce<<<(unsigned)((n_unique + 127) / 128), 128, 0, ctx->stream>>>(
          ctx->db, ctx->dp, ctx->dsets, ctx->dlut, ctx->dphase, ctx->dup_names ? 1 : 0, ctx->b_chunks.as<hm_chunk>(), ctx->b_pair_off.as<uint64_t>(),
          ctx->b_pair_hap.as<uint8_t>(), ctx->b_geom.as<int32_t>(), ctx->b_geom.as<int32_t>() + n_chunks, k_in, d_cnt + 1, site_lo,
          site_n, entries, stride, rec_buf.as<hm_site_record>(), d_cnt + 8, ctx->b_bidx.as<uint32_t>(),
          ctx->b_brecs.as<hm_site_record>(), (uint32_t)HM_BOUNDARY_CAP, d_cnt + 4, reinterpret_cast<int*>(d_cnt + 3), nullptr, nullptr, nullptr, 0,
          (uint32_t)HM_SITE_SLOTS);
      if (omit) { // records of germline restatements stay here: flags -> scan -> stable compaction
        CU(ctx->b_keep.ensure(n_unique * 4 + 16)); CU(ctx->b_kpos.ensure(n_unique * 4 + 16));
        CU(ctx->b_bpos.ensure(((size_t)HM_BOUNDARY_CAP + HM_BOUNDARY_FIRST) * 4));
        CU(ctx->b_compact[parity].ensure(n_unique * sizeof(hm_site_record)));
        const unsigned nb_ = (unsigned)((n_unique + 255) / 256);
        k_keep_flags<<<nb_, 256, 0, ctx->stream>>>(rec_buf.as<hm_site_record>(), d_cnt + 1, ctx->b_keep.as<uint32_t>());
        size_t tmp_scan = 0;
        CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp_scan, ctx->b_keep.as<uint32_t>(), ctx->b_kpos.as<uint32_t>(), (int64_t)n_unique, ctx->stream));
        if (tmp_scan > ctx->b_cub.cap) CU(ctx->b_cub.ensure(tmp_scan)); // the sort has finished with it (same stream)
        tmp_scan = ctx->b_cub.cap;
        CU(cub::DeviceScan::ExclusiveSum(ctx->b_cub.p, tmp_scan, ctx->b_keep.as<uint32_t>(), ctx->b_kpos.as<uint32_t>(), (int64_t)n_unique, ctx->stream));
        k_compact_records<<<nb_, 256, 0, ctx->stream>>>(rec_buf.as<hm_site_record>(), ctx->b_keep.as<uint32_t>(), ctx->b_kpos.as<uint32_t>(),
                                                      d_cnt + 1, ctx->b_compact[parity].as<hm_site_record>());
        k_gather_u32<<<8, 256, 0, ctx->stream>>>(ctx->b_kpos.as<uint32_t>(), ctx->b_bidx.as<uint32_t>(), d_cnt + 4, (uint32_t)HM_BOUNDARY_CAP,
                                                ctx->b_bpos.as<uint32_t>());
      }
      t_end(ctx);
      CU(cudaGetLastError());
    }
    t_begin(ctx, "k_count_flags");
    k_count_flags<<<148, 256, 0, ctx->stream>>>(ctx->b_qseen.as<uint8_t>(), (uint64_t)ctx->max_qname_id + 1, d_cnt + 2);
    t_end(ctx);
    CU(cudaGetLastError());
    // First the small things: counters and the boundary records (the only ones the sequential som_seen replay
    // looks at).  The big record copy follows the replay, so records a previous chunk already claimed are skipped
    // by the copy itself instead of being squeezed out of 20 MB on the host.
    k_publish<<<1, 64, 0, ctx->stream>>>(reinterpret_cast<const uint32_t*>(d_cnt), reinterpret_cast<uint32_t*>(ctx->h_cnt_pin), (uint32_t)(CNT_BYTES / 4));
    if (n_keys) {
      k_publish_items<<<4, 256, 0, ctx->stream>>>(ctx->b_bidx.as<uint32_t>(), h_bidx, 1u, (uint32_t)HM_BOUNDARY_FIRST, d_cnt + 4);
      k_publish_items<<<8, 256, 0, ctx->stream>>>(ctx->b_brecs.as<uint32_t>(), reinterpret_cast<uint32_t*>(h_brecs),
                                                  (uint32_t)(sizeof(hm_site_record) / 4), (uint32_t)HM_BOUNDARY_FIRST, d_cnt + 4);
      if (omit) k_publish_items<<<4, 256, 0, ctx->stream>>>(ctx->b_bpos.as<uint32_t>(), h_bpos, 1u, (uint32_t)HM_BOUNDARY_FIRST, d_cnt + 4);
    }
    CU(cudaGetLastError());
    lap(4); // site kernel launches enqueued
    CU(cudaStreamSynchronize(ctx->stream));
    lap(5); // sync 3: site kernels
    memcpy(h_cnt, ctx->h_cnt_pin, CNT_BYTES);
  }
  } // first version

  // ---- from here on both versions: counters are on the host, records still on the device ----
  size_t n_unique = (size_t)h_cnt[1], n_boundary = 0;
  // compacted: the records the host copies sit in b_compact (germline restatements left out when asked; the fused
  // path always compacts); boundary records are addressed through their
  // position there (h_bpos)
  const bool compacted = fused || omit;
  hm_site_record* recs = nullptr; // where the device records land on the host
  bool direct = false;
  bool have_all = false; // the records are already on the host (fallback of the boundary replay)
  struct Border { uint32_t idx, pos; hm_site_record rec; }; // index in key order, index among the kept records, the record
  std::vector<Border> border;
  unsigned long long* hist = h_cnt + 8;
  const size_t n_restate0 = (size_t)(hist[HM_ST_GERM_HET] + hist[HM_ST_GERM_HETALT] + hist[HM_ST_GERM_HOMALT] + hist[HM_ST_GERM_HOMREF]);
  if (n_pairs) {
    if ((int)h_cnt[3] == HM_ERR_BQ_ZERO) return fail(ctx, HM_ERR_BQ_ZERO, "a base quality of 0 reached the genotype model (the reference raises ValueError: math.log10(0))");
    n_boundary = n_keys ? (size_t)h_cnt[4] : 0;
    // records go straight into the caller's buffer when it is large enough, else into pinned staging
    {
      const size_t n_ret = fused ? (size_t)h_cnt[6] : (omit ? n_unique - n_restate0 : n_unique);
      const size_t n_host = n_boundary > HM_BOUNDARY_CAP ? n_unique : n_ret; // the host fallback of the replay fetches everything
      direct = out && cap >= n_host;
      if (n_host && !direct) {
        if (n_host > ctx->h_stage_cap) {
          if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
          ctx->h_stage = nullptr; ctx->h_stage_cap = 0;
          const size_t want = n_host + n_host / 4 + 1024;
          CU(cudaHostAlloc((void**)&ctx->h_stage, want * sizeof(hm_site_record), cudaHostAllocDefault));
          ctx->h_stage_cap = want;
        }
      }
      recs = n_unique ? (direct ? out : ctx->h_stage) : nullptr;
    }
    if (n_boundary > HM_BOUNDARY_CAP) {
      // heavily overlapping region lists: more boundary records than the device list holds.  Fetch everything and
      // find them on the host with the same test k_site_reduce applies.
      CU(cudaMemcpyAsync(recs, rec_buf.p, n_unique * sizeof(hm_site_record), cudaMemcpyDeviceToHost, ctx->stream));
      CU(cudaStreamSynchronize(ctx->stream));
      border.clear();
      for (size_t i = 0; i < n_unique; i++)
        if (recs[i].tpos <= prev_max_end[recs[i].chunk] || recs[i].tpos >= next_min_start[recs[i].chunk]) border.push_back(Border{(uint32_t)i, 0u, recs[i]});
      n_boundary = border.size();
      have_all = true;
    } else if (n_boundary) {
      border.resize(n_boundary);
      if (n_boundary <= (size_t)HM_BOUNDARY_FIRST) {
        for (size_t i = 0; i < n_boundary; i++) border[i] = Border{h_bidx[i], compacted ? h_bpos[i] : 0u, h_brecs[i]};
      } else {
        std::vector<uint32_t> bi(n_boundary), bp(n_boundary, 0u);
        std::vector<hm_site_record> br(n_boundary);
        CU(cudaMemcpyAsync(bi.data(), ctx->b_bidx.p, n_boundary * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(br.data(), ctx->b_brecs.p, n_boundary * sizeof(hm_site_record), cudaMemcpyDeviceToHost, ctx->stream));
        if (compacted) CU(cudaMemcpyAsync(bp.data(), ctx->b_bpos.p, n_boundary * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        for (size_t i = 0; i < n_boundary; i++) border[i] = Border{bi[i], bp[i], br[i]};
      }
    }
  }
  lap(6); // boundary list

  // sequential part: chunk order, som_seen carry (caller.py:324-347; bamlib.py:77), over the
  // boundary records only.  Indices are positions in the key order = (chunk, tpos, ref, alt).
  std::vector<uint32_t> dropped;
  // restatement records are counted before any of them is dropped by the replay
  const size_t n_restate = n_restate0;
  const bool in_compact = compacted && !have_all; // the copy below reads b_compact
  if (n_boundary) {
    std::sort(border.begin(), border.end(), [](const Border& a, const Border& b) { return a.idx < b.idx; });
    std::unordered_set<int32_t> som_seen;
    std::vector<int32_t> adds;
    size_t i = 0;
    while (i < n_boundary) {
      const int32_t chunk = border[i].rec.chunk;
      adds.clear();
      for (; i < n_boundary && border[i].rec.chunk == chunk; i++) {
        const hm_site_record& R = border[i].rec;
        const bool restates = R.status >= HM_ST_GERM_HET && R.status <= HM_ST_GERM_HOMREF;
        if (R.tpos <= prev_max_end[chunk] && som_seen.count(R.tpos)) { // dropped in get_tsbs_candidates
          if (!(in_compact && omit && restates)) dropped.push_back(in_compact ? border[i].pos : border[i].idx);
          hist[R.status]--;
          continue;
        }
        if (!restates && R.tpos >= next_min_start[chunk]) adds.push_back(R.tpos); // som_seen.add(tpos), caller.py:347
      }
      for (int32_t t : adds) som_seen.insert(t);
    }
    std::sort(dropped.begin(), dropped.end());
  }
  // what the copy below walks over: every record, or the compacted ones
  const size_t n_source = !in_compact ? n_unique : (fused ? (size_t)h_cnt[6] : n_unique - n_restate);
  const hm_site_record* d_source = in_compact ? ctx->b_compact[parity].as<hm_site_record>() : rec_buf.as<hm_site_record>();
  // the records, minus the dropped ones (ascending indices): one copy per run between two dropped records
  if ((rc = flush_deferred(ctx, false))) return rc; // an earlier call's copies, if this call had no sort to put them behind
  size_t n_final = 0;
  if (n_unique && have_all) {
    size_t from = 0;
    for (size_t d = 0; d <= dropped.size(); d++) {
      const size_t to = d < dropped.size() ? dropped[d] : n_unique;
      if (to > from && n_final != from) memmove(recs + n_final, recs + from, (to - from) * sizeof(hm_site_record));
      n_final += to - from;
      from = to + 1;
    }
    if (omit) { // the slow path has everything on the host: drop here what the compaction would have
      size_t w = 0;
      for (size_t i = 0; i < n_final; i++) {
        const uint8_t st = recs[i].status;
        if (omit && st >= HM_ST_GERM_HET && st <= HM_ST_GERM_HOMREF) continue;
        if (w != i) recs[w] = recs[i];
        w++;
      }
      n_final = w;
    }
  } else if (n_unique) {
    size_t from = 0;
    for (size_t d = 0; d <= dropped.size(); d++) {
      const size_t to = d < dropped.size() ? dropped[d] : n_source;
      if (to > from)
        ctx->deferred.push_back(hm_ctx::PendingCopy{recs + n_final, d_source + from, (to - from) * sizeof(hm_site_record)});
      n_final += to - from;
      from = to + 1;
    }
    ctx->deferred_parity = parity;
    ctx->rec_parity ^= 1;
    if (!async || !direct) { // copy now, behind whatever the main stream still has queued
      if ((rc = flush_deferred(ctx, true))) return rc;
      CU(cudaStreamSynchronize(ctx->copy_stream));
      ctx->copy_pending = false;
    }
  }
  t_collect(ctx);
  // chrom2tsbs_log (caller.py:625-641) from the status tallies
  {
    unsigned long long total = 0;
    for (int k = 0; k < 16; k++) total += hist[k];
    log[0] = (int64_t)h_cnt[2];
    log[1] = (int64_t)total;
    log[2] = (int64_t)hist[HM_ST_GERM_HET]; log[3] = (int64_t)hist[HM_ST_GERM_HETALT]; log[4] = (int64_t)hist[HM_ST_GERM_HOMALT];
    log[5] = (int64_t)(hist[HM_ST_HET_SITE] + hist[HM_ST_HETALT_SITE] + hist[HM_ST_HOMALT_SITE]);
    log[7] = (int64_t)hist[HM_ST_INDEL_SITE];
    log[8] = (int64_t)hist[HM_ST_LOW_GQ]; log[9] = (int64_t)hist[HM_ST_LOW_BQ]; log[10] = (int64_t)hist[HM_ST_PON];
    log[11] = (int64_t)hist[HM_ST_COMSNP]; log[12] = (int64_t)hist[HM_ST_HIGH_DEPTH]; log[13] = (int64_t)hist[HM_ST_LOW_DEPTH];
    log[14] = (int64_t)(hist[HM_ST_PASS] + hist[HM_ST_UNPHASED]); // num_som is counted before the phase verdict
    log[6] = log[8] + log[9] + log[10] + log[11] + log[12] + log[13] + log[14];
  }
  *n_out = n_final;
  lap(7); // host replay
  if (host_timing)
    fprintf(stderr, "[host timing, dev %d, %s] enqueue %.3f | sync1 %.3f | sort enqueue %.3f | sync2 %.3f | sites enqueue %.3f | sync3 %.3f | boundary %.3f | replay %.3f ms\n",
            ctx->device, fused ? "fused" : "first version", ht[0], ht[1], ht[2], ht[3], ht[4], ht[5], ht[6], ht[7]);
  if (!direct && n_final) {
    if (out && cap >= n_final) memcpy(out, recs, n_final * sizeof(hm_site_record));
    else {
      ctx->final_recs.assign(recs, recs + n_final);
      return fail(ctx, HM_ERR_CAPACITY, "output holds %zu records, %zu needed (hm_last_records fetches them without recomputing)", cap, n_final);
    }
  }
  return HM_OK;
}

/* records of the last hm_call_chunks that returned HM_ERR_CAPACITY, without recomputing */
int hm_last_records(hm_ctx* ctx, hm_site_record* out, size_t cap, size_t* n_out) {
  if (!ctx || !n_out) return HM_ERR_ARG;
  *n_out = ctx->final_recs.size();
  if (cap < ctx->final_recs.size() || (!out && !ctx->final_recs.empty())) return fail(ctx, HM_ERR_CAPACITY, "output holds %zu records, %zu needed", cap, ctx->final_recs.size());
  if (!ctx->final_recs.empty()) memcpy(out, ctx->final_recs.data(), ctx->final_recs.size() * sizeof(hm_site_record));
  return HM_OK;
}

int hm_call_batch(hm_ctx* ctx, const hm_read_batch* batch, const hm_chunk* chunks, size_t n_chunks, hm_site_record* out,
                  size_t cap, size_t* n_out, int64_t log[HM_CALL_LOG_LEN]) {
  int rc = hm_upload_batch(ctx, batch);
  if (rc) return rc;
  return hm_call_chunks(ctx, chunks, n_chunks, out, cap, n_out, log);
}

int hm_call_batch_compact(hm_ctx* ctx, const hm_read_batch* batch, const hm_bq_compact* bq, const hm_chunk* chunks, size_t n_chunks,
                          hm_site_record* out, size_t cap, size_t* n_out, int64_t log[HM_CALL_LOG_LEN]) {
  int rc = hm_upload_batch_compact(ctx, batch, bq);
  if (rc) return rc;
  return hm_call_chunks(ctx, chunks, n_chunks, out, cap, n_out, log);
}

int hm_read_stats(hm_ctx* ctx, int64_t* bq_total, int32_t* n_match, int32_t* n_sub, int32_t* ins_len, int32_t* del_len,
                  int32_t* n_mismatch) {
  if (!ctx) return HM_ERR_ARG;
  if (!ctx->have_params) return fail(ctx, HM_ERR_STATE, "hm_set_params has not been called");
  if (!ctx->have_batch) return fail(ctx, HM_ERR_STATE, "no resident batch");
  CU(cudaSetDevice(ctx->device));
  t_reset(ctx);
  int rc = launch_read_scan(ctx);
  if (rc) return rc;
  const size_t n = ctx->n_reads;
  static_assert(sizeof(unsigned long long) == sizeof(int64_t), "");
#define DN(dst, buf, T) if (dst && n) CU(cudaMemcpyAsync(dst, ctx->buf.p, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream))
  DN(bq_total, b_bq_total, int64_t); DN(n_match, b_n_match, int32_t); DN(n_sub, b_n_sub, int32_t);
  DN(ins_len, b_ins_len, int32_t); DN(del_len, b_del_len, int32_t); DN(n_mismatch, b_n_mm, int32_t);
#undef DN
  CU(cudaStreamSynchronize(ctx->stream));
  t_collect(ctx);
  return HM_OK;
}

int hm_normcounts_chunks(hm_ctx* ctx, const uint8_t* refseq, size_t ref_len, const hm_chunk* chunks, size_t n_chunks,
                         int64_t ccs_tri[HM_TRI_BINS], int64_t ref_tri[HM_TRI_BINS], int64_t log[HM_NORM_LOG_LEN],
                         int64_t* n_alt_tie) {
  int rc = check_ready(ctx, chunks, n_chunks);
  if (rc) return rc;
  return hm_normcounts_impl(ctx, refseq, ref_len, chunks, n_chunks, ccs_tri, ref_tri, log, n_alt_tie);
}

/* per-qname_id flags of the last call: 1 where some record with that id passed the read gates in
 * a chunk that fetched it (the reads m.num_ccs counts, caller.py:318-320) */
int hm_qname_seen(hm_ctx* ctx, uint8_t* out, size_t cap, size_t* n) {
  if (!ctx || !n) return HM_ERR_ARG;
  if (!ctx->have_batch) return fail(ctx, HM_ERR_STATE, "no resident batch");
  *n = (size_t)ctx->max_qname_id + 1;
  if (cap < *n || !out) return fail(ctx, HM_ERR_CAPACITY, "output holds %zu flags, %zu needed", cap, *n);
  CU(cudaSetDevice(ctx->device));
  if (ctx->b_qseen.cap < *n) return fail(ctx, HM_ERR_STATE, "no call has run on this batch yet");
  CU(cudaMemcpyAsync(out, ctx->b_qseen.p, *n, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return HM_OK;
}

/* keep a contig's reference sequence resident for subsequent hm_normcounts_chunks(refseq = NULL) */
int hm_set_reference(hm_ctx* ctx, const uint8_t* refseq, size_t ref_len) {
  if (!ctx || (!refseq && ref_len)) return HM_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  ctx->ref_len = 0;
  ctx->packed_pos = 0;
  int rc = upload(ctx, ctx->b_ref, refseq, ref_len);
  if (rc) return rc;
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->ref_len = ref_len;
  return HM_OK;
}

/* reference-genome trinucleotide counts of one contig (reflib.get_chrom_tricount) */
int hm_ref_tricounts(hm_ctx* ctx, const uint8_t* refseq, size_t ref_len, int64_t tri[HM_TRI_BINS]) {
  if (!ctx || !tri || (!refseq && ref_len)) return HM_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  memset(tri, 0, sizeof(int64_t) * HM_TRI_BINS);
  t_reset(ctx);
  int rc = upload(ctx, ctx->b_ref, refseq, ref_len);
  ctx->ref_len = 0;
  ctx->packed_pos = 0;
  if (rc) return rc;
  CU(ctx->b_norm_out.ensure(sizeof(NormOut)));
  CU(cudaMemsetAsync(ctx->b_norm_out.p, 0, sizeof(NormOut), ctx->stream));
  if (ref_len > 2) {
    t_begin(ctx, "k_ref_tricounts");
    k_ref_tricounts<<<148 * 8, 256, 0, ctx->stream>>>(ctx->b_ref.as<uint8_t>(), (uint64_t)ref_len, ctx->b_norm_out.as<NormOut>()->ccs_tri);
    t_end(ctx);
    CU(cudaGetLastError());
  }
  NormOut h;
  CU(cudaMemcpyAsync(&h, ctx->b_norm_out.p, sizeof(NormOut), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  t_collect(ctx);
  for (int i = 0; i < HM_TRI_BINS; i++) tri[i] = (int64_t)h.ccs_tri[i];
  return HM_OK;
}

/* how many positions the last hm_normcounts_chunks evaluated with the exact genotype arithmetic
 * (the rest were decided by the certified integer pass) */
int hm_last_norm_exact_sites(hm_ctx* ctx, uint64_t* n) {
  if (!ctx || !n) return HM_ERR_ARG;
  *n = (uint64_t)ctx->last_norm_sites;
  return HM_OK;
}

/* ---- `himut phase` edge counting (phaselib.get_edges) ---- */
int hm_phase_edges_begin(hm_ctx* ctx, const int32_t* hpos, const uint8_t* href, size_t n_hetsnp, uint32_t band) {
  if (!ctx || (n_hetsnp && (!hpos || !href)) || band == 0) return HM_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  for (size_t i = 1; i < n_hetsnp; i++) if (hpos[i - 1] > hpos[i]) return fail(ctx, HM_ERR_ARG, "hpos is not ascending");
  if ((uint64_t)n_hetsnp * band * 16 > (64ull << 30)) return fail(ctx, HM_ERR_ARG, "edge table of %zu x %u entries is too large", n_hetsnp, band);
  int rc;
  if ((rc = upload(ctx, ctx->b_edge_hpos, hpos, n_hetsnp))) return rc;
  if ((rc = upload(ctx, ctx->b_edge_href, href, n_hetsnp))) return rc;
  const size_t bytes = (size_t)n_hetsnp * band * 16 + 16;
  CU(ctx->b_edge_counts.ensure(bytes));
  CU(cudaMemsetAsync(ctx->b_edge_counts.p, 0, bytes, ctx->stream));
  CU(ctx->b_counters.ensure(256));
  CU(cudaMemsetAsync(ctx->b_counters.as<unsigned long long>() + 6, 0, 8, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->edge_n = n_hetsnp; ctx->edge_band = band;
  return HM_OK;
}

int hm_phase_edges_add(hm_ctx* ctx, int32_t min_bq, int32_t min_mapq, int32_t min_tstart, uint32_t* need_band) {
  if (!ctx || !need_band) return HM_ERR_ARG;
  if (!ctx->have_batch) return fail(ctx, HM_ERR_STATE, "no resident batch: call hm_upload_batch first");
  if (!ctx->edge_band) return fail(ctx, HM_ERR_STATE, "hm_phase_edges_begin has not been called");
  CU(cudaSetDevice(ctx->device));
  t_reset(ctx);
  int rc = launch_read_scan(ctx); // for its op prefixes; the read gates it also computes are not used here
  if (rc) return rc;
  unsigned int* d_need = reinterpret_cast<unsigned int*>(ctx->b_counters.as<unsigned long long>() + 6);
  if (ctx->n_reads && ctx->edge_n >= 2) {
    t_begin(ctx, "k_phase_edges");
    k_phase_edges<<<(unsigned)((ctx->n_reads * 32 + 127) / 128), 128, 0, ctx->stream>>>(
        ctx->db, ctx->b_edge_hpos.as<int32_t>(), ctx->b_edge_href.as<uint8_t>(), (uint32_t)ctx->edge_n, min_bq, min_mapq, min_tstart,
        ctx->edge_band, ctx->b_edge_counts.as<unsigned int>(), d_need);
    t_end(ctx);
    CU(cudaGetLastError());
  }
  unsigned int need = 0;
  CU(cudaMemcpyAsync(&need, d_need, 4, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  t_collect(ctx);
  *need_band = need;
  if (need == 0xffffffffu) return fail(ctx, HM_ERR_CAPACITY, "a read covers more than %d hetSNPs", HM_EDGE_MAX_SNPS);
  if (need > ctx->edge_band) return fail(ctx, HM_ERR_CAPACITY, "a read pairs hetSNPs %u apart in the list; the band is %u", need, ctx->edge_band);
  return HM_OK;
}

int hm_phase_edges_end(hm_ctx* ctx, uint32_t* counts, size_t cap_entries) {
  if (!ctx || !counts) return HM_ERR_ARG;
  if (!ctx->edge_band) return fail(ctx, HM_ERR_STATE, "hm_phase_edges_begin has not been called");
  const size_t n = (size_t)ctx->edge_n * ctx->edge_band * 4;
  if (cap_entries < n) return fail(ctx, HM_ERR_CAPACITY, "output holds %zu counters, %zu needed", cap_entries, n);
  CU(cudaSetDevice(ctx->device));
  if (n) CU(cudaMemcpyAsync(counts, ctx->b_edge_counts.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->edge_band = 0; ctx->edge_n = 0;
  return HM_OK;
}

int hm_last_timing(hm_ctx* ctx, float* total_ms, int* n_launches) {
  if (!ctx) return HM_ERR_ARG;
  if (total_ms) *total_ms = ctx->last_total_ms;
  if (n_launches) *n_launches = ctx->last_launches;
  return HM_OK;
}

int hm_last_call_path(hm_ctx* ctx) { return !ctx ? 0 : (ctx->call_path); }

int hm_last_kernel_times(hm_ctx* ctx, const char** names, float* ms, size_t cap, size_t* n) {
  if (!ctx || !n) return HM_ERR_ARG;
  size_t k = 0;
  for (; k < ctx->ktimes.size() && k < cap; k++) {
    if (names) names[k] = ctx->ktimes[k].name;
    if (ms) ms[k] = ctx->ktimes[k].ms;
  }
  *n = k;
  return HM_OK;
}

int hm_decode_bam_begin(hm_ctx* ctx, const hm_bgzf_plan* plan, int rid, int32_t start, int32_t end, uint64_t* n_reads) {
  return hm_decode_bam_begin_opts(ctx, plan, rid, start, end, 0, n_reads);
}

int hm_decode_bam_begin_opts(hm_ctx* ctx, const hm_bgzf_plan* plan, int rid, int32_t start, int32_t end, uint32_t opts,
                             uint64_t* n_reads) {
  if (!ctx || !plan || !n_reads) return HM_ERR_ARG;
  *n_reads = 0;
  if (opts & ~HM_DECODE_SEQ) return fail(ctx, HM_ERR_ARG, "unknown decode option bits 0x%x", opts & ~HM_DECODE_SEQ);
  CU(cudaSetDevice(ctx->device));
  if (ctx->upload_pending) { // the copies of an upload that was not waited for still read their host buffers
    CU(cudaEventSynchronize(ctx->ev_up));
    ctx->upload_pending = false;
  }
  ctx->have_batch = false;
  ctx->dec_ready = false;
  t_reset(ctx);
  if (start < 0) start = 0;
  const int rc = decode_begin_impl(ctx, plan, rid, start, end, (opts & HM_DECODE_SEQ) != 0, n_reads);
  if (rc) { cudaStreamSynchronize(ctx->stream); return rc; }
  t_collect(ctx);
  ctx->dec_ready = true;
  return HM_OK;
}

int hm_decode_bam_names(hm_ctx* ctx, const char** names, const uint64_t** name_off, const int32_t** tstart, const int32_t** tend,
                        uint64_t* n_reads) {
  if (!ctx || !names || !name_off || !tstart || !tend || !n_reads) return HM_ERR_ARG;
  if (!ctx->dec_ready) return fail(ctx, HM_ERR_STATE, "no decoded region: call hm_decode_bam_begin first");
  *names = ctx->hd_names.data(); *name_off = ctx->hd_name_off.data();
  *tstart = ctx->hd_tstart.data(); *tend = ctx->hd_tend.data();
  *n_reads = ctx->dec_n;
  return HM_OK;
}

int hm_decode_bam_end(hm_ctx* ctx, const uint32_t* qname_id) {
  if (!ctx) return HM_ERR_ARG;
  if (!ctx->dec_ready) return fail(ctx, HM_ERR_STATE, "no decoded region: call hm_decode_bam_begin first");
  const uint64_t n = ctx->dec_n;
  if (n && !qname_id) return fail(ctx, HM_ERR_ARG, "qname_id is NULL");
  CU(cudaSetDevice(ctx->device));
  ctx->dec_ready = false;
  ctx->hd_flags.assign(n, 0);
  const bool has_seq = ctx->dec_seq != 0;
  hm_read_batch b;
  memset(&b, 0, sizeof(b));
  b.n_reads = n;
  b.tstart = ctx->hd_tstart.data(); b.tend = ctx->hd_tend.data(); b.qstart = ctx->hd_qstart.data(); b.qlen = ctx->hd_qlen.data();
  b.flags = ctx->hd_flags.data(); b.qname_id = qname_id; b.bq_off = ctx->hd_bq_off.data(); b.op_off = ctx->hd_op_off.data();
  b.n_ops = ctx->hd_n_ops.data(); b.bq_bytes = ctx->dec_bq; b.n_ops_total = ctx->dec_ops;
  if (has_seq) { b.seq_off = ctx->hd_seq_off.data(); b.seq_bytes = ctx->dec_seq; }  // b.seq stays NULL: the stream is on the device
  int rc;
  if ((rc = batch_tables(ctx, &b, nullptr, has_seq))) return rc;
  if (n == 0) { // the host decoder's empty batch: 16 zero quality bytes (and 16 zero base bytes with the base stream)
    CU(ctx->b_bq.ensure(32));
    CU(cudaMemsetAsync(ctx->b_bq.p, 0, 16, ctx->stream));
    CU(ctx->b_ops.ensure(16));
    for (DevBuf* d : {&ctx->b_tstart, &ctx->b_tend, &ctx->b_qstart, &ctx->b_qlen, &ctx->b_mapq, &ctx->b_flags, &ctx->b_qname,
                      &ctx->b_n_ops, &ctx->b_bq_off, &ctx->b_op_off})
      CU(d->ensure(16));
    if (has_seq) {
      CU(ctx->b_seq.ensure(32));
      CU(cudaMemsetAsync(ctx->b_seq.p, 0, 16, ctx->stream));
      CU(ctx->b_seq_off.ensure(16));
    }
  }
  if ((rc = upload(ctx, ctx->b_qname, qname_id, n))) return rc;
  if ((rc = bind_batch(ctx, &b, has_seq))) return rc;
  if ((rc = launch_bq_sum(ctx))) return rc;
  ctx->compact_resident = false;
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->have_batch = true;
  return HM_OK;
}

/* diagnostics (tests): the resident batch back to caller buffers (NULL: skip); sizes as hm_decode_bam_begin / the upload
 * left them: n_reads entries per read, bq_bytes quality bytes, n_ops_total ops */
int hm_batch_read_back(hm_ctx* ctx, hm_read_batch* out, int32_t* tstart, int32_t* tend, int32_t* qstart, int32_t* qlen,
                       uint8_t* mapq, uint32_t* qname_id, uint64_t* bq_off, uint64_t* op_off, uint32_t* n_ops, uint8_t* bq, uint32_t* ops) {
  if (!ctx || !out) return HM_ERR_ARG;
  if (!ctx->have_batch) return fail(ctx, HM_ERR_STATE, "no resident batch");
  CU(cudaSetDevice(ctx->device));
  memset(out, 0, sizeof(*out));
  const uint64_t n = ctx->n_reads;
  out->n_reads = n; out->bq_bytes = ctx->bq_bytes; out->n_ops_total = ctx->n_ops_total;
  const struct { void* dst; const DevBuf* src; size_t bytes; } cp[] = {
      {tstart, &ctx->b_tstart, n * 4}, {tend, &ctx->b_tend, n * 4}, {qstart, &ctx->b_qstart, n * 4}, {qlen, &ctx->b_qlen, n * 4},
      {mapq, &ctx->b_mapq, n}, {qname_id, &ctx->b_qname, n * 4}, {bq_off, &ctx->b_bq_off, n * 8}, {op_off, &ctx->b_op_off, n * 8},
      {n_ops, &ctx->b_n_ops, n * 4}, {bq, &ctx->b_bq, ctx->bq_bytes}, {ops, &ctx->b_ops, ctx->n_ops_total * 4}};
  for (const auto& c : cp)
    if (c.dst && c.bytes) CU(cudaMemcpyAsync(c.dst, c.src->p, c.bytes, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return HM_OK;
}

/* diagnostics (tests): the resident base stream back to caller buffers (NULL: skip): n_reads offsets, *seq_bytes bytes;
 * *seq_bytes = 0 when the resident batch has no base stream */
int hm_batch_read_back_seq(hm_ctx* ctx, uint64_t* seq_off, uint8_t* seq, uint64_t* seq_bytes) {
  if (!ctx || !seq_bytes) return HM_ERR_ARG;
  if (!ctx->have_batch) return fail(ctx, HM_ERR_STATE, "no resident batch");
  *seq_bytes = ctx->db.seq ? ctx->seq_bytes : 0;
  if (!ctx->db.seq) return HM_OK;
  CU(cudaSetDevice(ctx->device));
  if (seq_off && ctx->n_reads) CU(cudaMemcpyAsync(seq_off, ctx->b_seq_off.p, ctx->n_reads * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (seq) CU(cudaMemcpyAsync(seq, ctx->b_seq.p, ctx->seq_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return HM_OK;
}

/* tests: k_bgzf_inflate's decoder on one raw DEFLATE stream that must inflate to exactly out_len bytes with CRC32 `crc`;
 * 0 ok, else the error code of bamerr.h (E_INFLATE, E_CRC) */
int hm_inflate_device_test(hm_ctx* ctx, const uint8_t* in, size_t in_len, uint8_t* out, size_t out_len, uint32_t crc) {
  if (!ctx || (in_len && !in) || (out_len && !out) || out_len > 65536 || in_len >= (1ull << 31)) return HM_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  DevBuf din, dout, drc;
  CU(din.ensure(in_len + 16));
  CU(dout.ensure(out_len + 16));
  CU(drc.ensure(16));
  if (in_len) CU(cudaMemcpyAsync(din.p, in, in_len, cudaMemcpyHostToDevice, ctx->stream));
  bamgpu::k_inflate_one<<<1, 32, 0, ctx->stream>>>(din.as<uint8_t>(), (uint32_t)in_len, dout.as<uint8_t>(), (uint32_t)out_len, crc, drc.as<int>());
  int rc = 0;
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(&rc, drc.p, 4, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess && out_len) e = cudaMemcpyAsync(out, dout.p, out_len, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  din.release(); dout.release(); drc.release();
  if (e != cudaSuccess) return fail(ctx, HM_ERR_CUDA, "hm_inflate_device_test: %s", cudaGetErrorString(e));
  return rc;
}

}  // extern "C"

static int hm_normcounts_impl(hm_ctx* ctx, const uint8_t* refseq, size_t ref_len, const hm_chunk* chunks, size_t n_chunks,
                              int64_t* ccs_tri, int64_t* ref_tri, int64_t* log, int64_t* n_alt_tie) {
  if (!ccs_tri || !ref_tri || !log) return fail(ctx, HM_ERR_ARG, "output pointer is NULL");
  if (!refseq && !ctx->ref_len) return fail(ctx, HM_ERR_STATE, "refseq is NULL and no reference was set with hm_set_reference");
  if (ctx->have_batch && !ctx->db.seq) return fail(ctx, HM_ERR_STATE, "the resident batch was uploaded without a base stream (seq == NULL): normcounts needs it");
  if (!refseq) ref_len = ctx->ref_len;
  CU(cudaSetDevice(ctx->device));
  memset(ccs_tri, 0, sizeof(int64_t) * HM_TRI_BINS);
  memset(ref_tri, 0, sizeof(int64_t) * HM_TRI_BINS);
  memset(log, 0, sizeof(int64_t) * HM_NORM_LOG_LEN);
  if (n_alt_tie) *n_alt_tie = 0;
  ctx->last_norm_sites = 0;
  t_reset(ctx);
  std::vector<uint64_t> pair_off;
  int rc = upload_chunks(ctx, chunks, n_chunks, pair_off);
  if (rc) return rc;
  const uint64_t n_pairs = pair_off.back();
  // tile prefix sums of k_norm_tiles_tma (512-position tiles from each chunk's start)
  std::vector<uint64_t> tile_off(n_chunks + 1, 0);
  for (size_t i = 0; i < n_chunks; i++) {
    const int64_t span = (int64_t)chunks[i].end - (int64_t)chunks[i].start;
    tile_off[i + 1] = tile_off[i] + (span > 0 ? (uint64_t)((span + HM_TW - 1) / HM_TW) : 0);
  }
  const uint64_t n_tiles = tile_off[n_chunks];
  if (n_tiles >= (1ull << 31)) return fail(ctx, HM_ERR_ARG, "too many tiles in one call");
  if ((rc = upload(ctx, ctx->b_tile_off, tile_off.data(), tile_off.size()))) return rc;
  if (refseq) { // per-call reference: replaces whatever hm_set_reference left
    if ((rc = upload(ctx, ctx->b_ref, refseq, ref_len))) return rc;
    ctx->ref_len = 0;
    ctx->packed_pos = 0;
  }
  // bit vectors (normbits.cuh) in front of the exact pass; the single pass k_norm_tiles_tma where they do not apply:
  // parameters outside the certified domain, a chunk that starts below 0 (the spans lie on the absolute 1024 grid),
  // cal words that a 32-bit offset cannot address
  bool use_bits = ctx->cert.enabled && ctx->n_reads > 0 && ctx->n_cw < (1ull << 32) && n_pairs > 0;
  std::vector<uint64_t> span_off(n_chunks + 1, 0);
  int64_t max_end = 0;
  for (size_t i = 0; i < n_chunks; i++) {
    const int64_t span = (int64_t)chunks[i].end - (int64_t)chunks[i].start;
    if (chunks[i].start < 0) use_bits = false;
    span_off[i + 1] = span_off[i] + (span > 0 && chunks[i].start >= 0 ? (uint64_t)(((chunks[i].end - 1) >> 10) - (chunks[i].start >> 10) + 1) : 0);
    max_end = std::max<int64_t>(max_end, chunks[i].end);
  }
  const uint64_t n_spans = span_off[n_chunks];
  uint64_t imp_words = 0;
  if (use_bits) {
    const uint64_t need_pos = std::max<uint64_t>(std::max<uint64_t>((uint64_t)ref_len, (uint64_t)std::max(ctx->h_pmax.back(), 0) + 2), (uint64_t)max_end);
    const uint64_t n_pos = (need_pos + 1023) / 1024 * 1024 + 1024;
    if (ctx->packed_pos < n_pos) {
      CU(ctx->b_ref2.ensure(n_pos / 4 + 16));
      CU(ctx->b_tri8.ensure(n_pos + 16));
      t_begin(ctx, "k_ref_pack");
      k_ref_pack<<<(unsigned)((n_pos / 16 + 255) / 256), 256, 0, ctx->stream>>>(ctx->b_ref.as<uint8_t>(), (uint64_t)ref_len, n_pos, ctx->b_ref2.as<uint32_t>(),
                                                                             ctx->b_tri8.as<uint8_t>());
      t_end(ctx);
      CU(cudaGetLastError());
      ctx->packed_pos = refseq ? 0 : n_pos; // a per-call reference is packed per call
    }
    imp_words = n_pos / 32;
    CU(ctx->b_impure.ensure(imp_words * 4 + 16));
    CU(cudaMemsetAsync(ctx->b_impure.p, 0, imp_words * 4, ctx->stream));
    CU(ctx->b_sdiff.ensure(imp_words * 4 + 16));
    CU(cudaMemsetAsync(ctx->b_sdiff.p, 0, imp_words * 4, ctx->stream));
    CU(ctx->b_cal_ok.ensure((size_t)ctx->n_reads + 16));
    CU(ctx->b_calw.ensure((size_t)ctx->n_cw * 4 + 16));
    if ((rc = upload(ctx, ctx->b_thr, ctx->cert_thr, 256))) return rc;
    if ((rc = upload(ctx, ctx->b_span_off, span_off.data(), span_off.size()))) return rc;
    t_begin(ctx, "k_norm_prep");
    k_norm_prep<<<(unsigned)((ctx->n_reads + NB_PREP_WARPS - 1) / NB_PREP_WARPS), 32 * NB_PREP_WARPS, sizeof(PrepWarp) * NB_PREP_WARPS, ctx->stream>>>(
        ctx->db, ctx->dp, ctx->b_ref2.as<uint32_t>(), ctx->b_cw_off.as<uint32_t>(), ctx->b_calw.as<uint32_t>(), ctx->b_impure.as<uint32_t>(), imp_words,
        ctx->compact_resident ? ctx->b_bqmask.as<uint16_t>() : nullptr, ctx->b_exc_minmax.as<uint8_t>(),
        ctx->modal, ctx->b_sdiff.as<uint32_t>(), ctx->b_cal_ok.as<uint8_t>());
    t_end(ctx);
    CU(cudaGetLastError());
  } else if ((rc = launch_read_scan(ctx))) return rc;
  CU(ctx->b_norm_out.ensure(sizeof(NormOut)));
  CU(ctx->b_counters.ensure(64));
  CU(ctx->b_qseen.ensure((size_t)ctx->max_qname_id + 1));
  CU(ctx->b_pair_hap.ensure(n_pairs + 16));
  CU(cudaMemsetAsync(ctx->b_norm_out.p, 0, sizeof(NormOut), ctx->stream));
  CU(cudaMemsetAsync(ctx->b_counters.p, 0, 64, ctx->stream));
  CU(cudaMemsetAsync(ctx->b_qseen.p, 0, (size_t)ctx->max_qname_id + 1, ctx->stream));
  NormOut h;
  memset(&h, 0, sizeof(h));
  unsigned long long h_cnt[4] = {0, 0, 0, 0};
  if (n_pairs && n_tiles) {
    unsigned blocks = (unsigned)((n_pairs * 32 + 255) / 256);
    t_begin(ctx, "k_pair_info");
    k_pair_info<<<blocks, 256, 0, ctx->stream>>>(ctx->db, ctx->dp, ctx->dphase, ctx->b_chunks.as<hm_chunk>(), (uint32_t)n_chunks,
                                                 ctx->b_pair_off.as<uint64_t>(), n_pairs, ctx->b_pair_hap.as<uint8_t>(),
                                                 ctx->b_qseen.as<uint8_t>());
    t_end(ctx);
    CU(cudaGetLastError());
    int n_sm = 148;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, ctx->device);
    if (!use_bits) {
      const size_t smem = sizeof(TileStage) * HM_NSTAGE;
      static bool attr_set = false;
      if (!attr_set) {
        CU(cudaFuncSetAttribute(k_norm_tiles_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
      }
      const unsigned grid = (unsigned)std::min<uint64_t>(n_tiles, (uint64_t)n_sm);
      t_begin(ctx, "k_norm_tiles_tma");
      k_norm_tiles_tma<<<grid, HM_TW + 32 * HM_NPROD, smem, ctx->stream>>>(ctx->db, ctx->dp, ctx->dsets, ctx->dlut, ctx->b_chunks.as<hm_chunk>(),
                                                                (uint32_t)n_chunks, ctx->b_pair_off.as<uint64_t>(),
                                                                ctx->b_pair_hap.as<uint8_t>(), ctx->b_tile_off.as<uint64_t>(),
                                                                (uint32_t)n_tiles, ctx->b_ref.as<uint8_t>(), (uint64_t)ref_len,
                                                                ctx->b_norm_out.as<NormOut>());
      t_end(ctx);
    } else {
      // bit-vector pass over every position, then the exact pass over the listed sites
      unsigned long long* d_nsites = ctx->b_counters.as<unsigned long long>() + 4;
      unsigned long long n_sites = 0;
      const double md = ctx->params.md_threshold;
      const int md_k = !(md == md) ? 256 : md < 0.0 ? 0 : md >= 255.0 ? 256 : (int)floor(md) + 1; // depth >= md_k <=> depth > md_threshold
      const unsigned bgrid = (unsigned)std::min<uint64_t>((n_spans + NB_BITS_WARPS - 1) / NB_BITS_WARPS, (uint64_t)n_sm * (ctx->params.phase ? 4 : 6));
      CU(ctx->b_tile_info.ensure((size_t)n_spans * 16 + 16));
      if (n_spans) {
        t_begin(ctx, "k_span_ranges");
        k_span_ranges<<<(unsigned)((n_spans + 255) / 256), 256, 0, ctx->stream>>>(ctx->db, ctx->b_chunks.as<hm_chunk>(), (uint32_t)n_chunks,
                                                                              ctx->b_span_off.as<uint64_t>(), n_spans, ctx->b_tile_info.as<uint4>());
        t_end(ctx);
        CU(cudaGetLastError());
        // every span leaves its 32 site words and its count; the counts are scanned and the keys written span by span:
        // the site list comes out in (chunk, position) order and in exactly the room it needs
        CU(ctx->b_push.ensure((size_t)n_spans * 128 + 16));
        CU(ctx->b_span_cnt.ensure(((size_t)n_spans + 1) * 8 + 16));
        uint32_t* span_cnt = ctx->b_span_cnt.as<uint32_t>();
        uint32_t* span_dst = span_cnt + n_spans;
        t_begin(ctx, "k_norm_bits");
        (ctx->params.phase ? k_norm_bits<true> : k_norm_bits<false>)<<<bgrid, 32 * NB_BITS_WARPS, 0, ctx->stream>>>(
            ctx->db, ctx->dp, ctx->b_thr.as<uint16_t>(), (int)ctx->cert.n_min, md_k, ctx->b_chunks.as<hm_chunk>(), (uint32_t)n_chunks,
            ctx->b_pair_off.as<uint64_t>(), ctx->b_pair_hap.as<uint8_t>(), ctx->b_tile_info.as<uint4>(), n_spans, ctx->b_cw_off.as<uint32_t>(),
            ctx->b_calw.as<uint32_t>(), ctx->b_impure.as<uint32_t>(), ctx->b_tri8.as<uint8_t>(), ctx->b_norm_out.as<NormOut>(),
            ctx->b_push.as<uint32_t>(), span_cnt);
        t_end(ctx);
        CU(cudaGetLastError());
        t_begin(ctx, "k_emit_sites");
        k_span_scan<<<1, 1024, 0, ctx->stream>>>(span_cnt, n_spans, span_dst, d_nsites);
        CU(cudaMemcpyAsync(&n_sites, d_nsites, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        CU(ctx->b_sites.ensure((size_t)std::max<unsigned long long>(n_sites, 1) * 8));
        if (n_sites)
          k_emit_sites<<<(unsigned)((n_spans * 32 + 255) / 256), 256, 0, ctx->stream>>>(ctx->b_tile_info.as<uint4>(), n_spans, ctx->b_push.as<uint32_t>(),
                                                                                     span_dst, ctx->b_sites.as<unsigned long long>());
        t_end(ctx);
        CU(cudaGetLastError());
      }
      ctx->last_norm_sites = n_sites;
      const unsigned long long* site_keys = ctx->b_sites.as<unsigned long long>();
      if (n_sites) {
        CU(ctx->b_koff.ensure((n_chunks + 2) * 4));
        k_chunk_key_ranges<<<(unsigned)((n_chunks + 1 + 127) / 128), 128, 0, ctx->stream>>>(site_keys, d_nsites, (uint32_t)n_chunks, ctx->b_koff.as<uint32_t>());
      }
      // sites per round of the exact pass: the entry table (slots x sites x 4 B) stays at 0.5 GB
      const uint32_t n_slots = ctx->site_slots; // as the call path: about twice the mean depth
      const unsigned long long SITE_BATCH = std::max<unsigned long long>(1ull << 16, (1ull << 27) / std::max<uint32_t>(n_slots, 1u));
      for (unsigned long long s0 = 0; s0 < n_sites; s0 += SITE_BATCH) {
        const uint64_t nb = (uint64_t)std::min<unsigned long long>(SITE_BATCH, n_sites - s0);
        const uint64_t stride = (nb + 31) & ~31ull;
        CU(ctx->b_agg.ensure(stride * n_slots * 4 + nb * 8));
        uint32_t* entries = ctx->b_agg.as<uint32_t>();
        uint32_t* site_lo = entries + stride * n_slots;
        uint32_t* site_n = site_lo + nb;
        const unsigned long long* keys = site_keys + s0;
        t_begin(ctx, "k_norm_site_range");
        k_norm_site_range<<<(unsigned)((nb + 255) / 256), 256, 0, ctx->stream>>>(ctx->db, ctx->b_chunks.as<hm_chunk>(), keys, nb, site_lo, site_n);
        t_end(ctx);
        t_begin(ctx, "k_norm_entries_bits");
        CU(cudaMemsetAsync(entries, 0xff, stride * n_slots * 4, ctx->stream));
        k_norm_entries_bits<<<(unsigned)((n_pairs * 32 + 255) / 256), 256, 0, ctx->stream>>>(
            ctx->db, ctx->dp, ctx->b_chunks.as<hm_chunk>(), (uint32_t)n_chunks, ctx->b_pair_off.as<uint64_t>(), n_pairs,
            ctx->b_pair_hap.as<uint8_t>(), site_keys, ctx->b_koff.as<uint32_t>(), (uint64_t)s0, nb, site_lo, site_n, entries, stride,
            ctx->b_cw_off.as<uint32_t>(), ctx->b_calw.as<uint32_t>(), ctx->b_cal_ok.as<uint8_t>(), ctx->b_sdiff.as<uint32_t>(),
            ctx->b_ref2.as<uint32_t>(), ctx->compact_resident ? ctx->b_bqmask.as<uint16_t>() : nullptr, ctx->modal, n_slots);
        t_end(ctx);
        t_begin(ctx, "k_norm_reduce");
        k_norm_reduce<<<(unsigned)((nb + 127) / 128), 128, 0, ctx->stream>>>(
            ctx->db, ctx->dp, ctx->dsets, ctx->dlut, ctx->b_chunks.as<hm_chunk>(), ctx->b_pair_off.as<uint64_t>(),
            ctx->b_pair_hap.as<uint8_t>(), keys, nb, site_lo, site_n, entries, stride, ctx->b_ref.as<uint8_t>(), (uint64_t)ref_len,
            ctx->b_norm_out.as<NormOut>(), n_slots);
        t_end(ctx);
        CU(cudaGetLastError());
      }
    }
    CU(cudaGetLastError());
    t_begin(ctx, "k_count_flags");
    k_count_flags<<<148, 256, 0, ctx->stream>>>(ctx->b_qseen.as<uint8_t>(), (uint64_t)ctx->max_qname_id + 1,
                                                ctx->b_counters.as<unsigned long long>() + 2);
    t_end(ctx);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(&h, ctx->b_norm_out.p, sizeof(NormOut), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(h_cnt, ctx->b_counters.p, 32, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CU(cudaStreamSynchronize(ctx->stream));
  t_collect(ctx);
  if (h.err == HM_ERR_BQ_ZERO) return fail(ctx, HM_ERR_BQ_ZERO, "a base quality of 0 reached the genotype model (the reference raises ValueError: math.log10(0))");
  for (int i = 0; i < HM_TRI_BINS; i++) { ccs_tri[i] = (int64_t)h.ccs_tri[i]; ref_tri[i] = (int64_t)h.ref_tri[i]; }
  for (int i = 1; i < HM_NORM_LOG_LEN; i++) log[i] = (int64_t)h.log[i];
  log[0] = (int64_t)h_cnt[2];
  if (n_alt_tie) *n_alt_tie = (int64_t)h.alt_tie;
  return HM_OK;
}
