// normtrack.cuh — the callable-base track of `himut normcounts` as runs (HM_OPT_CALLABLE_TRACK).
//
// The normcounts kernels (k_norm_bits, k_norm_reduce, k_norm_tiles_tma) leave one uint32 per position of every chunk:
// the callable count of a counted position, 0 elsewhere (track_at, normcounts.cuh).  Two passes turn that into runs
// (chunk, start, end, value) — maximal ranges of consecutive counted positions of one chunk with one value — in chunk
// order, then position order, as the exact pass's site list is built (k_span_scan / k_emit_sites):
//
//   k_track_count  one warp per piece of 1024 positions of a chunk, lane = 32 positions: how many runs begin and how
//                  many end in the piece (a run may span pieces; it never spans chunks);
//   k_span_scan    (normbits.cuh) scans both counts: the k-th run to begin is the k-th run to end;
//   k_track_emit   the same warps write (chunk, start, value) at the rank of each beginning and `end` at the rank of
//                  each end: 16-byte records, in order, in exactly the room they need.
#pragma once
#include "normbits.cuh"

// the piece's chunk, its first track slot and the lane's 32 values, with the values just before and after them
struct TrackLane {
  uint32_t c;
  int32_t pos0;      // position of the lane's first value
  uint32_t v[32];
  uint32_t prev, next;
};

__device__ __forceinline__ void track_lane(const uint32_t* track, const uint64_t* track_off, const uint64_t* piece_off,
                                           uint32_t n_chunks, const hm_chunk* chunks, uint64_t piece, int lane, TrackLane& t) {
  t.c = upper_bound_dev(piece_off, n_chunks + 1, piece) - 1;
  const uint64_t t0 = __ldg(track_off + t.c), t1 = __ldg(track_off + t.c + 1); // the chunk's slots (a multiple of 32)
  const uint64_t l0 = (piece - __ldg(piece_off + t.c)) * NB_SPAN + 32u * (uint64_t)lane; // the lane's first slot in the chunk
  t.pos0 = (int32_t)((int64_t)chunks[t.c].start + (int64_t)l0);
  const bool on = t0 + l0 < t1;
  const uint4* src = reinterpret_cast<const uint4*>(track + t0 + l0); // t0, l0: multiples of 32
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const uint4 q = on ? __ldg(src + i) : make_uint4(0u, 0u, 0u, 0u);
    t.v[4 * i] = q.x; t.v[4 * i + 1] = q.y; t.v[4 * i + 2] = q.z; t.v[4 * i + 3] = q.w;
  }
  // neighbours: the lanes beside it; at the piece's edges the slot beyond it if it belongs to the same chunk, else 0
  t.prev = __shfl_up_sync(HM_FULL, t.v[31], 1);
  t.next = __shfl_down_sync(HM_FULL, t.v[0], 1);
  if (lane == 0) t.prev = l0 > 0 ? __ldg(track + t0 + l0 - 1) : 0u;
  if (lane == 31) t.next = t0 + l0 + 32 < t1 ? __ldg(track + t0 + l0 + 32) : 0u;
}

// bit i: a run begins (begin) / ends (end) at the lane's value i
__device__ __forceinline__ void track_edges(const TrackLane& t, uint32_t* begin, uint32_t* end) {
  uint32_t b = 0, e = 0;
#pragma unroll
  for (int i = 0; i < 32; i++) {
    const uint32_t v = t.v[i], before = i == 0 ? t.prev : t.v[i - 1], after = i == 31 ? t.next : t.v[i + 1];
    b |= (uint32_t)(v != 0u && v != before) << i;
    e |= (uint32_t)(v != 0u && v != after) << i;
  }
  *begin = b; *end = e;
}

__global__ void __launch_bounds__(256) k_track_count(const uint32_t* track, const uint64_t* track_off, const uint64_t* piece_off,
                                                     uint32_t n_chunks, const hm_chunk* chunks, uint64_t n_pieces,
                                                     uint32_t* begin_cnt, uint32_t* end_cnt) {
  const uint64_t piece = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (piece >= n_pieces) return;
  TrackLane t;
  track_lane(track, track_off, piece_off, n_chunks, chunks, piece, lane, t);
  uint32_t b, e;
  track_edges(t, &b, &e);
  const uint32_t nb = __reduce_add_sync(HM_FULL, (uint32_t)__popc(b)), ne = __reduce_add_sync(HM_FULL, (uint32_t)__popc(e));
  if (lane == 0) { begin_cnt[piece] = nb; end_cnt[piece] = ne; }
}

// runs: hm_callable_run as 4 words (chunk, start, end, value)
__global__ void __launch_bounds__(256) k_track_emit(const uint32_t* track, const uint64_t* track_off, const uint64_t* piece_off,
                                                    uint32_t n_chunks, const hm_chunk* chunks, uint64_t n_pieces,
                                                    const uint32_t* begin_dst, const uint32_t* end_dst, uint32_t* runs) {
  const uint64_t piece = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (piece >= n_pieces) return;
  if (__ldg(begin_dst + piece + 1) == __ldg(begin_dst + piece) && __ldg(end_dst + piece + 1) == __ldg(end_dst + piece)) return;
  TrackLane t;
  track_lane(track, track_off, piece_off, n_chunks, chunks, piece, lane, t);
  uint32_t b, e;
  track_edges(t, &b, &e);
  uint32_t ib = (uint32_t)__popc(b), ie = (uint32_t)__popc(e);
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t x = __shfl_up_sync(HM_FULL, ib, d), y = __shfl_up_sync(HM_FULL, ie, d);
    if (lane >= d) { ib += x; ie += y; }
  }
  uint64_t at_b = (uint64_t)__ldg(begin_dst + piece) + ib - (uint32_t)__popc(b);
  uint64_t at_e = (uint64_t)__ldg(end_dst + piece) + ie - (uint32_t)__popc(e);
  while (b) {
    const int i = __ffs(b) - 1;
    b &= b - 1;
    uint32_t* r = runs + 4 * at_b++;
    *reinterpret_cast<uint2*>(r) = make_uint2(t.c, (uint32_t)(t.pos0 + i));
    r[3] = t.v[i];
  }
  while (e) {
    const int i = __ffs(e) - 1;
    e &= e - 1;
    runs[4 * at_e++ + 2] = (uint32_t)(int32_t)((int64_t)t.pos0 + i + 1); // <= ch.end: no wrap at 2^31 - 1
  }
}
