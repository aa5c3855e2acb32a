// bamgpu.cuh — a BAM region decoded on the device, from the compressed BGZF blocks to a resident batch with one
// quality byte per base: without a base stream for `call` and the phase edges, with the 2-bit base stream for
// normcounts.  The rules are hm_bam_read_batch's (csrc/bamdec.c), which stays the reference the tests compare against;
// the messages come from the same table (bamerr.h).
//
//   k_bgzf_inflate   one thread per BGZF block: raw DEFLATE (stored, fixed, dynamic), ISIZE and CRC32 checked
//   k_bam_walk       one thread per entry point (BAI linear-index entry): follows block_size to the next one
//   k_bam_select     one thread per record: hm_bam_read_batch's selection and checks, counts for the output scans
//   k_bam_parse      one warp per selected record: qualities, 2-bit bases (if asked), cs -> ops, coordinates, the name
//
// Shape of k_bgzf_inflate: a BGZF block is an independent stream of at most 64 KB whose decode is one serial chain
// (each symbol's length is known only once it is decoded), so one thread decodes one block, and it is the only
// thread of its warp: lanes that decode different streams diverge at every symbol.  Huffman codes are decoded
// canonically (count / symbol tables of 16 + 288 entries per code, zlib's puff.c) from local memory.
#pragma once
#include <cstdint>

#include "bamerr.h"

namespace bamgpu {

struct Plan {  // device copy of hm_bgzf_plan
  const uint8_t* comp;
  const uint64_t* coff;
  const uint32_t* csize;
  const uint32_t* isize;
  const uint64_t* uoff;
  const uint32_t* crc;
  uint64_t n_blocks;
};

struct Err {                    // first failure, in file order, of each kind
  unsigned long long block;     // first BGZF block that fails (~0: none); its code in blk_code
  unsigned long long entry;     // first entry point that is not a record start (~0: none)
  unsigned long long rec;       // first record that fails selection (~0: none)
  unsigned long long stop;      // first record that ends the region (~0: none)
  unsigned long long parse;     // first selected record that fails cs -> ops (~0: none)
};

struct RecInfo {  // k_bam_select -> k_bam_parse
  uint64_t p;     // offset of block_size in the inflated stream
  uint32_t cs;    // offset of the cs:Z value from the fixed part
  int32_t pos, l_seq, lead, trail, ref_span;
  uint32_t n_ops;
  uint8_t keep;
};

__device__ __forceinline__ uint32_t rd32(const uint8_t* p) {
  return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

// ------------------------------------------------------------------------------------------ k_bgzf_inflate
__constant__ uint16_t c_lbase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_lext[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t c_dbase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t c_dext[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__constant__ uint8_t c_clorder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct Bits {
  const uint8_t* p;
  uint32_t pos, len;
  uint64_t bb;
  int bc;
  bool err;
  // the next n (<= 32) bits; reading past the block's compressed payload is an error, never a read
  __device__ __forceinline__ uint32_t get(int n) {
    while (bc < n) {
      if (pos >= len) { err = true; return 0; }
      bb |= (uint64_t)p[pos++] << bc;
      bc += 8;
    }
    const uint32_t v = (uint32_t)(bb & ((1ull << n) - 1));
    bb >>= n;
    bc -= n;
    return v;
  }
};

struct Huff {
  int16_t count[16];
  int16_t sym[288];
};

// canonical code of n symbols from their lengths: < 0 over-subscribed, > 0 incomplete, 0 complete
__device__ int huff_build(Huff& h, const uint8_t* len, int n) {
  for (int i = 0; i < 16; i++) h.count[i] = 0;
  for (int s = 0; s < n; s++) h.count[len[s]]++;
  if (h.count[0] == n) return 0;
  int left = 1;
  for (int l = 1; l < 16; l++) {
    left <<= 1;
    left -= h.count[l];
    if (left < 0) return left;
  }
  int16_t offs[16];
  offs[1] = 0;
  for (int l = 1; l < 15; l++) offs[l + 1] = (int16_t)(offs[l] + h.count[l]);
  for (int s = 0; s < n; s++)
    if (len[s]) h.sym[offs[len[s]]++] = (int16_t)s;
  return left;
}

__device__ __forceinline__ int huff_decode(Bits& b, const Huff& h) {
  int code = 0, first = 0, index = 0;
  for (int l = 1; l < 16; l++) {
    code |= (int)b.get(1);
    if (b.err) return -1;
    const int cnt = h.count[l];
    if (code - cnt < first) return h.sym[index + (code - first)];
    index += cnt;
    first += cnt;
    first <<= 1;
    code <<= 1;
  }
  return -1;  // a code the table does not have
}

// one raw DEFLATE stream into out[0, isize): 0 ok, E_INFLATE (bad stream, wrong size), E_CRC
__device__ int inflate_block(const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t isize, uint32_t want_crc,
                             bool check_crc, const uint32_t* crc_tab) {
  Bits b{in, 0, in_len, 0ull, 0, false};
  Huff lit, dist;
  uint8_t lens[320];
  uint32_t n = 0, crc = 0xffffffffu;
  int last;
  do {
    last = (int)b.get(1);
    const uint32_t type = b.get(2);
    if (b.err) return E_INFLATE;
    if (type == 0) {  // stored
      b.bb >>= (b.bc & 7);
      b.bc -= (b.bc & 7);
      const uint32_t ln = b.get(16), nln = b.get(16);
      if (b.err || ln != (~nln & 0xffffu) || n + ln > isize) return E_INFLATE;
      for (uint32_t k = 0; k < ln; k++) {
        const uint8_t v = (uint8_t)b.get(8);
        if (b.err) return E_INFLATE;
        out[n++] = v;
        crc = crc_tab[(crc ^ v) & 0xff] ^ (crc >> 8);
      }
      continue;
    }
    if (type == 1) {  // fixed codes
      for (int s = 0; s < 144; s++) lens[s] = 8;
      for (int s = 144; s < 256; s++) lens[s] = 9;
      for (int s = 256; s < 280; s++) lens[s] = 7;
      for (int s = 280; s < 288; s++) lens[s] = 8;
      huff_build(lit, lens, 288);
      for (int s = 0; s < 30; s++) lens[s] = 5;
      huff_build(dist, lens, 30);
    } else if (type == 2) {  // dynamic codes
      const int nlen = (int)b.get(5) + 257, ndist = (int)b.get(5) + 1, ncode = (int)b.get(4) + 4;
      if (b.err || nlen > 286 || ndist > 30) return E_INFLATE;
      for (int k = 0; k < 19; k++) lens[c_clorder[k]] = k < ncode ? (uint8_t)b.get(3) : 0;
      if (b.err || huff_build(lit, lens, 19) != 0) return E_INFLATE;  // the code-length code must be complete
      int k = 0;
      while (k < nlen + ndist) {
        const int s = huff_decode(b, lit);
        if (s < 0) return E_INFLATE;
        if (s < 16) { lens[k++] = (uint8_t)s; continue; }
        uint8_t v = 0;
        int rep;
        if (s == 16) {
          if (k == 0) return E_INFLATE;
          v = lens[k - 1];
          rep = 3 + (int)b.get(2);
        } else if (s == 17) rep = 3 + (int)b.get(3);
        else rep = 11 + (int)b.get(7);
        if (b.err || k + rep > nlen + ndist) return E_INFLATE;
        while (rep--) lens[k++] = v;
      }
      if (lens[256] == 0) return E_INFLATE;  // no end-of-block code
      int e = huff_build(lit, lens, nlen);
      if (e < 0 || (e > 0 && nlen - lit.count[0] != 1)) return E_INFLATE;
      e = huff_build(dist, lens + nlen, ndist);
      if (e < 0 || (e > 0 && ndist - dist.count[0] != 1)) return E_INFLATE;
    } else return E_INFLATE;
    for (;;) {
      int s = huff_decode(b, lit);
      if (s < 0) return E_INFLATE;
      if (s < 256) {
        if (n >= isize) return E_INFLATE;
        out[n++] = (uint8_t)s;
        crc = crc_tab[(crc ^ (uint32_t)s) & 0xff] ^ (crc >> 8);
        continue;
      }
      if (s == 256) break;
      s -= 257;
      if (s >= 29) return E_INFLATE;
      const uint32_t len = c_lbase[s] + b.get(c_lext[s]);
      const int ds = huff_decode(b, dist);
      if (ds < 0 || ds >= 30) return E_INFLATE;
      const uint32_t d = c_dbase[ds] + b.get(c_dext[ds]);
      if (b.err || d > n || n + len > isize) return E_INFLATE;  // no reach before the block's start, no write past ISIZE
      const uint8_t* src = out + n - d;
      for (uint32_t k = 0; k < len; k++) {
        const uint8_t v = src[k];
        out[n + k] = v;
        crc = crc_tab[(crc ^ v) & 0xff] ^ (crc >> 8);
      }
      n += len;
    }
  } while (!last);
  if (n != isize) return E_INFLATE;
  if (check_crc && (crc ^ 0xffffffffu) != want_crc) return E_CRC;
  return 0;
}

__device__ __forceinline__ void crc_table_to_smem(uint32_t* tab) {
  for (int i = threadIdx.x; i < 256; i += blockDim.x) {
    uint32_t c = (uint32_t)i;
    for (int k = 0; k < 8; k++) c = (c & 1) ? 0xedb88320u ^ (c >> 1) : c >> 1;
    tab[i] = c;
  }
  __syncthreads();
}

// blocks [per_cta * blockIdx.x, +per_cta) of the plan, one per thread
__global__ void k_bgzf_inflate(Plan pl, uint8_t* out, uint32_t per_cta, uint8_t* blk_code, Err* err) {
  __shared__ uint32_t crc_tab[256];
  crc_table_to_smem(crc_tab);
  if (threadIdx.x >= per_cta) return;
  const uint64_t i = (uint64_t)blockIdx.x * per_cta + threadIdx.x;
  if (i >= pl.n_blocks) return;
  const uint8_t* h = pl.comp + pl.coff[i];
  const uint32_t csize = pl.csize[i], isize = pl.isize[i];
  const uint32_t xlen = (uint32_t)h[10] | ((uint32_t)h[11] << 8);  // inside the block: the host walked its header
  const int rc = csize < 12 + xlen + 8 ? E_INFLATE : inflate_block(h + 12 + xlen, csize - 12 - xlen - 8, out + pl.uoff[i], isize, pl.crc[i], true, crc_tab);
  if (rc) {
    blk_code[i] = (uint8_t)rc;
    atomicMin(&err->block, (unsigned long long)i);
  }
}

// one raw stream (tests): *rc = 0 or the code
__global__ void k_inflate_one(const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t out_len, uint32_t crc, int* rc) {
  __shared__ uint32_t crc_tab[256];
  crc_table_to_smem(crc_tab);
  if (threadIdx.x == 0) *rc = inflate_block(in, in_len, out, out_len, crc, true, crc_tab);
}

// ------------------------------------------------------------------------------------------ k_bam_walk
// Entry point e starts a segment that ends at the next entry point (the last one at walk_end).  Counting pass
// (offs == nullptr): cnt[e] = records of the segment; writing pass: their offsets at rec[seg_off[e]...].  A record
// that runs over the next entry point means the index does not point at record starts.  In the last segment a record
// that runs past walk_end is kept (k_bam_select reports it as truncated, in file order) and fewer than 4 bytes left
// are the end of the data, as the host decoder reads them.
__global__ void k_bam_walk(const uint8_t* buf, const uint64_t* entry, uint64_t n_entry, uint64_t walk_end,
                           unsigned long long* cnt, const unsigned long long* seg_off, uint64_t* rec, Err* err) {
  const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_entry) return;
  const bool last = e + 1 == n_entry;
  const uint64_t lim = last ? walk_end : entry[e + 1];
  uint64_t p = entry[e], k = 0, w = seg_off ? seg_off[e] : 0;
  while (p < lim) {
    if (lim - p < 4) {
      if (!last) atomicMin(&err->entry, (unsigned long long)(e + 1));
      break;
    }
    const uint64_t next = p + 4 + rd32(buf + p);
    if (next > lim && !last) { atomicMin(&err->entry, (unsigned long long)(e + 1)); break; }
    if (rec) rec[w + k] = p;
    k++;
    if (next > lim) break;
    p = next;
  }
  if (cnt) cnt[e] = k;
}

// ------------------------------------------------------------------------------------------ k_bam_select
// counts per record for the exclusive scans: [0] selected, [1] ops, [2] quality bytes (16-byte padded), [3] name bytes,
// and with the base stream (n_cnt 5) [4] its bytes, ceil(l_seq / 4) padded to 16 as the host decoder lays them out
__device__ __forceinline__ void sel_fail(Err* err, uint8_t* code, long long* arg, uint64_t r, int c, long long a) {
  code[r] = (uint8_t)c;
  arg[r] = a;
  atomicMin(&err->rec, (unsigned long long)r);
}

// ops the cs string gives (the ':0' token gives none); stops where the grammar of k_bam_parse would fail
__device__ uint32_t cs_count(const char* c) {
  uint32_t n = 0;
  while (*c) {
    if (*c == ':') {
      c++;
      if (*c < '0' || *c > '9') break;
      bool nz = false;
      while (*c >= '0' && *c <= '9') { nz |= *c != '0'; c++; }
      n += nz;
    } else if (*c == '=' || *c == '+' || *c == '-') {
      c++;
      const char* s = c;
      while ((*c >= 'A' && *c <= 'Z') || (*c >= 'a' && *c <= 'z')) c++;
      if (c == s) break;
      n++;
    } else if (*c == '*') {
      if (!c[1] || !c[2]) break;
      c += 3;
      n++;
    } else break;
  }
  return n;
}

__global__ void k_bam_select(const uint8_t* buf, const uint64_t* rec, uint64_t n_rec, uint64_t walk_end, int32_t rid,
                             int32_t start, int32_t end, RecInfo* info, unsigned long long* cnt, int n_cnt, uint8_t* code,
                             long long* arg, Err* err) {
  const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t stride = n_rec + 1;  // cnt: n_cnt (4 or 5) arrays of n_rec + 1 (the last entry 0: the scan's total)
  if (r == 0)
    for (int k = 0; k < n_cnt; k++) cnt[k * stride + n_rec] = 0;
  if (r >= n_rec) return;
  for (int k = 0; k < n_cnt; k++) cnt[k * stride + r] = 0;
  RecInfo I;
  I.keep = 0;
  I.p = rec[r];
  const uint32_t bs = rd32(buf + I.p);
  if (I.p + 4 + (uint64_t)bs > walk_end) { info[r] = I; sel_fail(err, code, arg, r, E_TRUNC_REC, 0); return; }
  const uint8_t* R = buf + I.p + 4;
  const int32_t ref_id = (int32_t)rd32(R), pos = (int32_t)rd32(R + 4);
  info[r] = I;
  if (ref_id != rid) {
    if (ref_id > rid || ref_id < 0) atomicMin(&err->stop, (unsigned long long)r);
    return;
  }
  if (pos >= end) { atomicMin(&err->stop, (unsigned long long)r); return; }
  if (bs < 32) { sel_fail(err, code, arg, r, E_BLOCK_SIZE, bs); return; }
  const uint32_t l_name = R[8], n_cig = R[12] | (R[13] << 8), flag = R[14] | (R[15] << 8);
  const int32_t l_seq = (int32_t)rd32(R + 16);
  if (l_seq < 0 || l_name == 0 || 32 + (uint64_t)l_name + 4 * (uint64_t)n_cig + ((uint64_t)l_seq + 1) / 2 + (uint64_t)l_seq > (uint64_t)bs ||
      R[32 + l_name - 1] != 0) {
    sel_fail(err, code, arg, r, E_FIELDS, bs);
    return;
  }
  const uint8_t* cig = R + 32 + l_name;
  int32_t ref_span = 0, lead = 0, trail = 0;
  for (uint32_t k = 0; k < n_cig; k++) {
    const uint32_t c = rd32(cig + 4 * k), op = c & 15, ln = c >> 4;
    if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) ref_span += (int32_t)ln;
  }
  for (uint32_t k = 0; k < n_cig; k++) { const uint32_t c = rd32(cig + 4 * k), op = c & 15; if (op == 4) lead += (int32_t)(c >> 4); else if (op != 5) break; }
  for (uint32_t k = n_cig; k-- > 0;) { const uint32_t c = rd32(cig + 4 * k), op = c & 15; if (op == 4) trail += (int32_t)(c >> 4); else if (op != 5) break; }
  const int32_t rend = pos + (ref_span > 0 ? ref_span : 1);
  if (rend <= start) return;
  if (flag & 0x100) return;
  const uint8_t* seq4 = cig + 4 * (size_t)n_cig;
  const uint8_t* qual = seq4 + ((size_t)l_seq + 1) / 2;
  const uint8_t* tag = qual + (l_seq > 0 ? l_seq : 0);
  const uint8_t* rec_end = R + bs;
  const uint8_t* cs = nullptr;
  while (tag + 3 <= rec_end) {
    const char ty = (char)tag[2];
    const uint8_t* v = tag + 3;
    const size_t left = (size_t)(rec_end - v);
    size_t adv;
    if (ty == 'Z' || ty == 'H') {
      size_t z = 0;
      while (z < left && v[z]) z++;
      if (z == left) { sel_fail(err, code, arg, r, E_TAG_UNTERM, ty); return; }
      adv = z + 1;
      if (tag[0] == 'c' && tag[1] == 's' && ty == 'Z') cs = v;
    } else if (ty == 'A' || ty == 'c' || ty == 'C') adv = 1;
    else if (ty == 's' || ty == 'S') adv = 2;
    else if (ty == 'i' || ty == 'I' || ty == 'f') adv = 4;
    else if (ty == 'B') {
      if (left < 5) { sel_fail(err, code, arg, r, E_TAG_B, (long long)left); return; }
      const char sub = (char)v[0];
      const uint32_t cnt = rd32(v + 1);
      adv = 5 + (size_t)cnt * ((sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : 4);
    } else { sel_fail(err, code, arg, r, E_TAG_TYPE, ty); return; }
    if (adv > left) { sel_fail(err, code, arg, r, E_TAG_PAST, (long long)adv); return; }
    tag = v + adv;
  }
  if (!cs) { sel_fail(err, code, arg, r, E_NO_CS, 0); return; }
  if (l_seq <= 0 || qual[0] == 0xff) { sel_fail(err, code, arg, r, E_NO_QUAL, 0); return; }
  I.keep = 1;
  I.cs = (uint32_t)(cs - R);
  I.pos = pos; I.l_seq = l_seq; I.lead = lead; I.trail = trail; I.ref_span = ref_span;
  I.n_ops = cs_count((const char*)cs);
  info[r] = I;
  cnt[r] = 1;
  cnt[stride + r] = I.n_ops;
  cnt[2 * stride + r] = ((uint64_t)l_seq + 15) & ~(uint64_t)15;
  cnt[3 * stride + r] = l_name;
  if (n_cnt == 5) cnt[4 * stride + r] = (((uint64_t)l_seq + 3) / 4 + 15) & ~(uint64_t)15;
}

// ------------------------------------------------------------------------------------------ k_bam_parse
struct ParseOut {
  int32_t *tstart, *tend, *qstart, *qlen;
  uint8_t *mapq, *flags;
  uint32_t* n_ops;
  uint64_t *bq_off, *op_off, *name_off;
  uint8_t* bq;
  uint32_t* ops;
  char* names;
  uint64_t* seq_off;  // both nullptr: no base stream (the batch of `call` and the phase edges)
  uint8_t* seq;
};

// the code of read base q (A0 T1 G2 C3, 0xff anything else)
__device__ __forceinline__ uint8_t base_at(const uint8_t* seq4, int64_t q) {
  const int8_t nib2code[16] = {-1, 0, 3, -1, 2, -1, -1, -1, 1, -1, -1, -1, -1, -1, -1, -1};
  const uint8_t by = seq4[q >> 1];
  return (uint8_t)nib2code[(q & 1) ? (by & 15) : (by >> 4)];
}
__device__ __forceinline__ int base_code(char c) {
  switch (c) { case 'A': case 'a': return 0; case 'T': case 't': return 1; case 'G': case 'g': return 2; case 'C': case 'c': return 3; default: return -1; }
}

// 2-bit code of each BAM nibble at bits 2 * nibble: A (1) 0, C (2) 3, G (4) 2, T (8) 1; N, IUPAC codes and '=' 0, as
// the host decoder's pack_codes_* store them
constexpr uint32_t kNibBits = (3u << 2 * 2) | (2u << 2 * 4) | (1u << 2 * 8);

// Every lane of the warp walks the cs string (the same bytes: broadcast loads, no divergence); checks over a run of
// read bases are split over the lanes, and lane 0 writes the ops.  scan: exclusive prefix sums of k_bam_select's
// counts (stride apart) = the record's read index and its first op, quality byte, name byte and (o.seq) base byte.
// n_rec: the records before the one that ends the region.
__global__ void k_bam_parse(const uint8_t* buf, const RecInfo* info, uint64_t n_rec, const unsigned long long* scan,
                            uint64_t stride, ParseOut o, uint8_t* code, long long* arg, Err* err) {
  const uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= n_rec) return;
  const RecInfo I = info[r];
  if (!I.keep) return;
  const uint64_t rd = scan[r], op0 = scan[stride + r], bq0 = scan[2 * stride + r], nm0 = scan[3 * stride + r];
  const uint8_t* R = buf + I.p + 4;
  const uint32_t l_name = R[8], n_cig = R[12] | (R[13] << 8);
  const int32_t l_seq = I.l_seq;
  const uint8_t* seq4 = R + 32 + l_name + 4 * (size_t)n_cig;
  const uint8_t* qual = seq4 + ((size_t)l_seq + 1) / 2;
  const uint64_t qb16 = ((uint64_t)l_seq + 15) & ~(uint64_t)15;
  for (uint64_t k = lane; k < qb16; k += 32) o.bq[bq0 + k] = k < (uint64_t)l_seq ? qual[k] : 0;
  for (uint32_t k = lane; k < l_name; k += 32) o.names[nm0 + k] = (char)R[32 + k];
  const uint64_t sq0 = o.seq ? scan[4 * stride + r] : 0;
  if (o.seq) {  // a lane packs 16 bases (8 nibble bytes) into one aligned word: base 16 w + j at bits 2 j of word w
    const uint64_t n_words = ((((uint64_t)l_seq + 3) / 4 + 15) & ~(uint64_t)15) / 4;  // the padding words are zero
    uint32_t* dst = (uint32_t*)(o.seq + sq0);
    for (uint64_t w = lane; w < n_words; w += 32) {
      const int64_t b0 = 16 * (int64_t)w, nb = min((int64_t)16, (int64_t)l_seq - b0);
      uint32_t v = 0;
      for (int64_t j = 0; j < nb; j += 2) {  // the high nibble is the even base
        const uint32_t by = seq4[(b0 + j) >> 1];
        v |= ((kNibBits >> 2 * (by >> 4)) & 3u) << 2 * j;
        if (j + 1 < nb) v |= ((kNibBits >> 2 * (by & 15)) & 3u) << 2 * (j + 1);
      }
      dst[w] = v;
    }
  }
  const char* cs = (const char*)(R + I.cs);
  const char* c = cs;
  uint32_t* ops = o.ops + op0;
  uint32_t n_ops = 0;
  int64_t q = I.lead, rspan = 0;
  int ec = 0;
  long long ea = 0;
  while (*c && !ec) {
    if (*c == ':') {
      long long n = 0;
      c++;
      if (*c < '0' || *c > '9') { ec = E_CS_TOKEN; ea = c - cs; break; }
      while (*c >= '0' && *c <= '9') { n = n * 10 + (*c++ - '0'); if (n > l_seq) { ec = E_CS_PAST; ea = n; break; } }
      if (ec) break;
      if (q + n > l_seq) { ec = E_CS_PAST; ea = q + n; break; }
      for (int64_t k0 = 0; k0 < n; k0 += 32) {  // first base outside A/C/G/T under the match
        const bool bad = k0 + lane < n && base_at(seq4, q + k0 + lane) == 0xff;
        const unsigned m = __ballot_sync(0xffffffffu, bad);
        if (m) { ec = E_N_MATCH; ea = q + k0 + __ffs(m) - 1; break; }
      }
      if (ec) break;
      if (n) { if (lane == 0 && n_ops < I.n_ops) ops[n_ops] = HM_MAKE_OP(HM_OP_MATCH, (uint32_t)n); n_ops++; }
      q += n; rspan += n;
    } else if (*c == '=') {
      long long n = 0;
      c++;
      while ((c[n] >= 'A' && c[n] <= 'Z') || (c[n] >= 'a' && c[n] <= 'z')) n++;
      if (n == 0 || q + n > l_seq) { ec = E_CS_TOKEN; ea = c - cs; break; }
      for (int64_t k0 = 0; k0 < n; k0 += 32) {  // first long-form base that is not the read's
        bool bad = false;
        if (k0 + lane < n) { const int bc = base_code(c[k0 + lane]); bad = bc < 0 || base_at(seq4, q + k0 + lane) != (uint8_t)bc; }
        const unsigned m = __ballot_sync(0xffffffffu, bad);
        if (m) { ec = E_CS_LONG; ea = q + k0 + __ffs(m) - 1; break; }
      }
      if (ec) break;
      if (lane == 0 && n_ops < I.n_ops) ops[n_ops] = HM_MAKE_OP(HM_OP_MATCH, (uint32_t)n);
      n_ops++;
      c += n; q += n; rspan += n;
    } else if (*c == '*') {
      if (!c[1] || !c[2]) { ec = E_CS_TOKEN; ea = c - cs; break; }
      const int rc_ = base_code(c[1]), ac = base_code(c[2]);
      if (ac < 0) { ec = E_SUB_N; ea = q; break; }
      if (lane == 0 && n_ops < I.n_ops) ops[n_ops] = HM_MAKE_SUB(rc_ < 0 ? HM_BASE_N : (uint32_t)rc_, (uint32_t)ac);
      n_ops++;
      c += 3; q += 1; rspan += 1;
    } else if (*c == '+' || *c == '-') {
      const bool ins = *c == '+';
      long long n = 0;
      c++;
      while ((c[n] >= 'A' && c[n] <= 'Z') || (c[n] >= 'a' && c[n] <= 'z')) n++;
      if (n == 0) { ec = E_CS_TOKEN; ea = c - cs; break; }
      if (lane == 0 && n_ops < I.n_ops) ops[n_ops] = HM_MAKE_OP(ins ? HM_OP_INS : HM_OP_DEL, (uint32_t)n);
      n_ops++;
      c += n;
      if (ins) q += n; else rspan += n;
    } else { ec = E_CS_TOKEN; ea = c - cs; break; }
  }
  if (!ec && rspan != I.ref_span) { ec = E_SPAN_REF; ea = rspan; }
  if (!ec && q - I.lead != (int64_t)l_seq - I.trail - I.lead) { ec = E_SPAN_QRY; ea = q - I.lead; }
  if (!ec && n_ops != I.n_ops) { ec = E_CS_TOKEN; ea = c - cs; }  // k_bam_select counted with the same grammar
  if (lane != 0) return;
  if (ec) {
    code[r] = (uint8_t)ec;
    arg[r] = ea;
    atomicMin(&err->parse, (unsigned long long)r);
    return;
  }
  o.tstart[rd] = I.pos;
  o.tend[rd] = I.pos + (int32_t)rspan;
  o.qstart[rd] = I.lead;
  o.qlen[rd] = l_seq;
  o.mapq[rd] = R[9];
  o.flags[rd] = 0;
  o.n_ops[rd] = n_ops;
  o.bq_off[rd] = bq0;
  o.op_off[rd] = op0;
  o.name_off[rd] = nm0;
  if (o.seq) o.seq_off[rd] = sq0;
}

}  // namespace bamgpu
