// Deterministic dedup (stable radix sort + segment boundaries) and the segment-reduce fused with the
// embedding row update (dense-grad / SGD / lazy Adam).  Replaces autograd's embedding_dense_backward and
// optimizer.step() for embedding tables (reference trainer/trainer.py:38-39).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/iterator/counting_input_iterator.cuh>
#include <cub/iterator/transform_input_iterator.cuh>

#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "segment.cuh"

namespace {
using rs::UpdParams;
using rs::upd_sgd;
using rs::adam1;

struct Offsets {
  int64_t off[RS_MAX_FIELDS];
};

// Padding (p >= *n_valid) gets the key `pad_key` = one past the largest real key: it sorts behind every real lookup and is
// then ignored by all the kernels below, which stop at *n_valid.
__global__ void __launch_bounds__(256) make_keys_kernel(const int64_t *__restrict__ ids, int64_t n, int F, const __grid_constant__ Offsets O,
                                                       int64_t total_rows, uint32_t *__restrict__ keys, int32_t *__restrict__ pos,
                                                       int32_t *status, const int32_t *__restrict__ n_valid, int shard_world,
                                                       int64_t shard_rows, uint32_t pad_key, int32_t *__restrict__ scalars,
                                                       int32_t *__restrict__ seg_start) {
  __shared__ int64_t s_off[RS_MAX_FIELDS + 1];
  for (int i = threadIdx.x; i < F; i += blockDim.x) s_off[i] = O.off[i];
  if (threadIdx.x == 0) s_off[F] = total_rows;
  __syncthreads();
  int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p == 0) {   // the device scalars (n_uniq, n_chunks, n_multi, work counter) start at zero: an empty (all padding) list
    scalars[0] = scalars[1] = scalars[2] = scalars[3] = 0;   // then leaves n_uniq = n_chunks = 0 and seg_start[0] = 0
    seg_start[0] = 0;
  }
  if (p >= n) return;
  pos[p] = (int32_t)p;
  if (n_valid && p >= *n_valid) {
    keys[p] = pad_key;
    return;
  }
  int f = (int)(p % F);
  int64_t lo = s_off[f];
  int64_t hi = (f + 1 < F ? s_off[f + 1] : total_rows);
  int64_t id = rs::clamp_id(ids[p], hi - lo, status);
  int64_t g = lo + id;
  if (shard_world > 1) g = (g % shard_world) * shard_rows + g / shard_world;   // owner-major: owner * R + local index
  keys[p] = (uint32_t)g;
}

#define RS_NV(nvp, n) ((nvp) ? (int64_t) * (nvp) : (n))   /* number of real (non-padding) lookups */

// head of a segment / of a chunk, recomputed where needed instead of being stored (nv = number of real lookups)
__device__ __forceinline__ bool is_head(const uint32_t *__restrict__ k, int64_t s, int64_t nv) {
  return s < nv && (s == 0 || k[s] != k[s - 1]);
}
__device__ __forceinline__ bool is_chunk_head(const int32_t *__restrict__ segidx1, const int32_t *__restrict__ seg_start, int64_t s,
                                              int64_t nv) {
  return s < nv && (((int)s - seg_start[segidx1[s] - 1]) % RS_CHUNK) == 0;
}
// scan inputs computed on the fly (cub::TransformInputIterator over a counting iterator)
struct HeadOp {
  const uint32_t *k;
  const int32_t *nvp;
  int64_t n;
  __device__ __forceinline__ int32_t operator()(int32_t s) const { return is_head(k, s, RS_NV(nvp, n)) ? 1 : 0; }
};
struct ChunkHeadOp {
  const int32_t *segidx1, *seg_start, *nvp;
  int64_t n;
  __device__ __forceinline__ int32_t operator()(int32_t s) const { return is_chunk_head(segidx1, seg_start, s, RS_NV(nvp, n)) ? 1 : 0; }
};

__global__ void __launch_bounds__(256) head_flags_kernel(const uint32_t *__restrict__ k, int64_t n, int32_t *__restrict__ head,
                                                        const int32_t *__restrict__ nvp) {
  int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  head[s] = (s < RS_NV(nvp, n) && (s == 0 || k[s] != k[s - 1])) ? 1 : 0;
}

// segidx1 = inclusive scan of head flags (1-based segment index)
__global__ void __launch_bounds__(256) seg_scatter_kernel(const uint32_t *__restrict__ k, const int32_t *__restrict__ pos,
                                                         const int32_t *__restrict__ segidx1, int64_t n,
                                                         int64_t *__restrict__ uniq, int32_t *__restrict__ seg_start,
                                                         int32_t *__restrict__ inverse, int32_t *__restrict__ n_uniq,
                                                         const int32_t *__restrict__ nvp) {
  int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  n = RS_NV(nvp, n);
  if (s >= n) return;
  int g = segidx1[s] - 1;
  if (is_head(k, s, n)) {
    uniq[g] = (int64_t)k[s];
    seg_start[g] = (int32_t)s;
  }
  inverse[pos[s]] = g;
  if (s == n - 1) {
    *n_uniq = g + 1;
    seg_start[g + 1] = (int32_t)n;
  }
}

// (only the hand-written scan of sort.cu needs the flags in memory; the cub path scans them on the fly)
__global__ void __launch_bounds__(256) chunk_flags_kernel(const int32_t *__restrict__ segidx1, const int32_t *__restrict__ seg_start,
                                                         int64_t n, int32_t *__restrict__ chead, const int32_t *__restrict__ nvp) {
  int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  chead[s] = is_chunk_head(segidx1, seg_start, s, RS_NV(nvp, n)) ? 1 : 0;
}

__global__ void __launch_bounds__(256) chunk_scatter_kernel(const int32_t *__restrict__ segidx1, const int32_t *__restrict__ seg_start,
                                                           const int32_t *__restrict__ chunkidx1,
                                                           int64_t n, int32_t *__restrict__ chunk_start, int32_t *__restrict__ chunk_seg,
                                                           int32_t *__restrict__ seg_first_chunk, int32_t *__restrict__ n_chunks,
                                                           int32_t *__restrict__ counts, const int32_t *__restrict__ nvp) {
  int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  n = RS_NV(nvp, n);
  if (s >= n) return;
  int g = segidx1[s] - 1;
  int c = chunkidx1[s] - 1;
  const int st = seg_start[g];
  if ((((int)s - st) % RS_CHUNK) == 0) {          // chunk head
    chunk_start[c] = (int32_t)s;
    chunk_seg[c] = g;
    if ((int)s == st) {                           // segment head
      seg_first_chunk[g] = c;
      counts[g] = seg_start[g + 1] - st;
    }
  }
  if (s == n - 1) {
    *n_chunks = c + 1;
    chunk_start[c + 1] = (int32_t)n;
    seg_first_chunk[g + 1] = c + 1;
  }
}

// Last pass, three independent jobs in one launch:
//  (a) segments cut into more than one chunk need a second pass; list them (order is irrelevant to the numerics);
//  (b) one 16-byte record per sorted lookup so the streaming update kernel needs a single coalesced read per lookup
//      instead of chasing chunk -> segment -> row through three arrays;
//  (c) work units of the streaming kernel start on chunk boundaries: unit u = chunks whose first lookup is in
//      [u*RS_UNIT, (u+1)*RS_UNIT).  unit_start[u] = first chunk start >= u*RS_UNIT (n past the end).
__global__ void __launch_bounds__(256) dedup_finish_kernel(const int32_t *__restrict__ sorted_pos, const int32_t *__restrict__ segidx1,
                                                          const int32_t *__restrict__ chunkidx1, const int32_t *__restrict__ seg_start,
                                                          const int32_t *__restrict__ chunk_start, const int32_t *__restrict__ chunk_seg,
                                                          const int32_t *__restrict__ seg_first_chunk, const int64_t *__restrict__ uniq,
                                                          int64_t n, int nunits, int4 *__restrict__ desc, int32_t *__restrict__ unit_start,
                                                          const int32_t *__restrict__ n_uniq, int32_t *__restrict__ multi_seg,
                                                          int32_t *__restrict__ n_multi, const int32_t *__restrict__ nvp) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nv = RS_NV(nvp, n);
  if (s < *n_uniq && seg_first_chunk[s + 1] - seg_first_chunk[s] > 1) multi_seg[atomicAdd(n_multi, 1)] = (int32_t)s;     // (a)
  if (s < n) {                                                                                                           // (b)
    if (s >= nv) {
      desc[s] = make_int4(0, 0, 0, 0);
    } else {
      const int c = chunkidx1[s] - 1;
      const int s0 = chunk_start[c], s1 = chunk_start[c + 1];
      const int g = chunk_seg[c];
      const bool single = (seg_first_chunk[g + 1] - seg_first_chunk[g]) == 1;
      int flags = (s == s0 ? 1 : 0) | (s + 1 == s1 ? 2 : 0) | (single ? 4 : 0);
      desc[s] = make_int4(sorted_pos[s], flags, (int)(uint32_t)uniq[g], 2 * (s0 / RS_CHUNK) + ((s1 - s0) < RS_CHUNK ? 1 : 0));
    }
  }
  if (s <= nunits) {                                                                                                     // (c)
    int64_t t = s * RS_UNIT;
    while (t < nv && !is_chunk_head(segidx1, seg_start, t, nv)) ++t;   // a chunk has at most RS_CHUNK lookups: stops within RS_CHUNK steps
    unit_start[s] = (int32_t)(t < nv ? t : nv);
  }
}

// Rename the rows of a finished sort to their rank among the distinct keys (row of segment g := g).
__global__ void __launch_bounds__(256) relabel_kernel(int4 *__restrict__ desc, const int32_t *__restrict__ inverse,
                                                     int64_t *__restrict__ uniq, const int32_t *__restrict__ n_uniq, int64_t n) {
  int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  desc[s].z = inverse[desc[s].x];
  if (s < *n_uniq) uniq[s] = s;
}

}  // namespace
namespace rs {   // sort.cu
size_t radix_sort_ws_ints(int64_t n);
size_t scan_ws_ints(int64_t n);
int radix_sort_pairs(const uint32_t *kin, const int32_t *vin, uint32_t *kout, int32_t *vout, uint32_t *ktmp, int32_t *vtmp,
                     int32_t *hist_ws, int64_t n, int end_bit, cudaStream_t st);
int inclusive_sum_i32(const int32_t *in, int32_t *out, int64_t n, int32_t *ws, cudaStream_t st);
}  // namespace rs
namespace {

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

struct WsLayout {
  size_t sorted_key, sorted_pos, uniq, inverse, counts, seg_start, seg_first_chunk, chunk_start, chunk_seg, multi_seg, lookup_desc, unit_start, scale_sorted, scalars;
  size_t keys_in, pos_in, head, segidx1, chead, chunkidx1, cub, sort_hist, scan_ws, partial, total;
  size_t cub_bytes, partial_floats;
};

WsLayout layout(int64_t n, int max_width) {
  WsLayout L;
  size_t o = 0;
  auto take = [&](size_t bytes) {
    size_t at = o;
    o += align_up(bytes);
    return at;
  };
  size_t n1 = (size_t)n + 1;
  L.sorted_key = take(n * 4);
  L.sorted_pos = take(n * 4);
  L.uniq = take(n * 8);
  L.inverse = take(n * 4);
  L.counts = take(n * 4);
  L.seg_start = take(n1 * 4);
  L.seg_first_chunk = take(n1 * 4);
  L.chunk_start = take(n1 * 4);
  L.chunk_seg = take(n * 4);
  L.multi_seg = take(n * 4);
  L.lookup_desc = take(n * 16);
  L.unit_start = take((n / RS_UNIT + 2) * 4);
  L.scale_sorted = take(n * 4);
  L.scalars = take(64);
  L.keys_in = take(n * 4);
  L.pos_in = take(n * 4);
  L.head = take(n * 4);
  L.segidx1 = take(n * 4);
  L.chead = take(n * 4);
  L.chunkidx1 = take(n * 4);
  size_t sort_b = 0, scan_b = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort_b, (const uint32_t *)nullptr, (uint32_t *)nullptr, (const int32_t *)nullptr,
                                  (int32_t *)nullptr, (int)n, 0, 32);
  cub::DeviceScan::InclusiveSum(nullptr, scan_b, (const int32_t *)nullptr, (int32_t *)nullptr, (int)n);
  {
    using Count = cub::CountingInputIterator<int32_t>;
    size_t b1 = 0, b2 = 0;
    cub::TransformInputIterator<int32_t, HeadOp, Count> heads(Count(0), HeadOp{nullptr, nullptr, n});
    cub::TransformInputIterator<int32_t, ChunkHeadOp, Count> cheads(Count(0), ChunkHeadOp{nullptr, nullptr, nullptr, n});
    cub::DeviceScan::InclusiveSum(nullptr, b1, heads, (int32_t *)nullptr, (int)n);
    cub::DeviceScan::InclusiveSum(nullptr, b2, cheads, (int32_t *)nullptr, (int)n);
    scan_b = scan_b > b1 ? scan_b : b1;
    scan_b = scan_b > b2 ? scan_b : b2;
  }
  L.cub_bytes = sort_b > scan_b ? sort_b : scan_b;
  L.cub = take(L.cub_bytes);
  L.sort_hist = take(rs::radix_sort_ws_ints(n) * 4);   // per-tile digit counts of the hand-written radix sort
  L.scan_ws = take(rs::scan_ws_ints(n) * 4);
  // Only chunks of multi-chunk segments store a partial.  Such chunks are all full (RS_CHUNK lookups) except the
  // tail of each segment, so slot = 2*(chunk_start/RS_CHUNK) + is_tail is injective and < 2*(n/RS_CHUNK + 1)
  // (see partial_slot below).
  L.partial_floats = (size_t)(2 * (n / RS_CHUNK + 2)) * (size_t)max_width;
  L.partial = take(L.partial_floats * 4);
  L.total = o;
  return L;
}

}  // namespace

RS_API int rs_dedup_workspace_bytes(int64_t n, int32_t max_width, size_t *bytes) {
  RS_CHECK_ARG(bytes && n >= 0 && n < (1ll << 31) && max_width >= 1, RS_E_ARG, "rs_dedup_workspace_bytes: bad argument");
  *bytes = layout(n > 0 ? n : 1, max_width).total;
  return RS_OK;
}

RS_API int rs_dedup_sort(const int64_t *ids, int64_t n, int32_t F, const int64_t *row_offset, int64_t total_rows, void *ws,
                         size_t ws_bytes, rs_segments *seg, int32_t *status, void *stream) {
  return rs_dedup_sort_ex(ids, n, F, row_offset, total_rows, nullptr, ws, ws_bytes, seg, status, stream);
}

RS_API int rs_dedup_sort_ex(const int64_t *ids, int64_t n, int32_t F, const int64_t *row_offset, int64_t total_rows,
                            const rs_dedup_opts *opts, void *ws, size_t ws_bytes, rs_segments *seg, int32_t *status, void *stream) {
  RS_CHECK_ARG(ids && ws && seg, RS_E_ARG, "rs_dedup_sort: null argument");
  const int32_t *nvp = opts ? opts->n_valid : nullptr;
  const int shard_world = opts ? opts->shard_world : 0;
  const int64_t shard_rows = opts ? opts->shard_rows : 0;
  int64_t key_space = total_rows;                  // keys live in [0, key_space)
  if (shard_world > 1) {
    RS_CHECK_ARG(shard_rows >= (total_rows + shard_world - 1) / shard_world, RS_E_ARG, "rs_dedup_sort_ex: shard_rows too small");
    key_space = (int64_t)shard_world * shard_rows;
  }
  if (nvp) key_space += 1;                         // the padding key
  RS_CHECK_ARG(key_space < (1ll << 32), RS_E_SHAPE, "rs_dedup_sort_ex: key space must be < 2^32");
  RS_CHECK_ARG(n > 0 && n < (1ll << 31), RS_E_SHAPE, "rs_dedup_sort: n must be in [1, 2^31)");
  RS_CHECK_ARG(F >= 1 && F <= RS_MAX_FIELDS && n % F == 0, RS_E_SHAPE, "rs_dedup_sort: bad F");
  RS_CHECK_ARG(total_rows > 0 && total_rows < (1ll << 32), RS_E_SHAPE, "rs_dedup_sort: total_rows must be < 2^32");
  // recover max_width from the workspace size is not possible; the caller sized ws with its own max_width, so
  // recompute the layout with width 1 for the fixed part and give the remainder to the partial buffer.
  WsLayout L = layout(n, 1);
  RS_CHECK_ARG(ws_bytes >= L.total, RS_E_WORKSPACE, "rs_dedup_sort: workspace too small (%zu < %zu)", ws_bytes, L.total);
  char *w = (char *)ws;
  seg->sorted_key = (uint32_t *)(w + L.sorted_key);
  seg->sorted_pos = (int32_t *)(w + L.sorted_pos);
  seg->uniq = (int64_t *)(w + L.uniq);
  seg->inverse = (int32_t *)(w + L.inverse);
  seg->counts = (int32_t *)(w + L.counts);
  seg->seg_start = (int32_t *)(w + L.seg_start);
  seg->seg_first_chunk = (int32_t *)(w + L.seg_first_chunk);
  seg->chunk_start = (int32_t *)(w + L.chunk_start);
  seg->chunk_seg = (int32_t *)(w + L.chunk_seg);
  seg->multi_seg = (int32_t *)(w + L.multi_seg);
  seg->n_uniq = (int32_t *)(w + L.scalars);
  seg->n_chunks = seg->n_uniq + 1;
  seg->n_multi = seg->n_uniq + 2;
  seg->work_counter = seg->n_uniq + 3;
  seg->lookup_desc = (int32_t *)(w + L.lookup_desc);
  seg->unit_start = (int32_t *)(w + L.unit_start);
  seg->scale_sorted = (float *)(w + L.scale_sorted);
  seg->partial = (float *)(w + L.partial);
  seg->partial_floats = (int64_t)((ws_bytes - L.partial) / 4);
  uint32_t *keys_in = (uint32_t *)(w + L.keys_in);
  int32_t *pos_in = (int32_t *)(w + L.pos_in);
  int32_t *head = (int32_t *)(w + L.head);
  int32_t *segidx1 = (int32_t *)(w + L.segidx1);
  int32_t *chead = (int32_t *)(w + L.chead);
  int32_t *chunkidx1 = (int32_t *)(w + L.chunkidx1);
  void *cub_ws = w + L.cub;
  size_t cub_bytes = L.cub_bytes;

  Offsets O;
  for (int f = 0; f < RS_MAX_FIELDS; ++f) O.off[f] = (row_offset && f < F) ? row_offset[f] : 0;
  if (!row_offset) RS_CHECK_ARG(F == 1, RS_E_ARG, "rs_dedup_sort: row_offset required when F > 1");
  cudaStream_t st = (cudaStream_t)stream;
  int blocks = (int)((n + 255) / 256);
  make_keys_kernel<<<blocks, 256, 0, st>>>(ids, n, F, O, total_rows, keys_in, pos_in, status, nvp, shard_world, shard_rows,
                                           (uint32_t)(key_space - 1), seg->n_uniq, seg->seg_start);
  RS_CHECK_LAUNCH();
  int end_bit = 1;
  while (end_bit < 32 && (1ull << end_bit) < (uint64_t)key_space) ++end_bit;
  // Stable sort by row key.  Default: cub::DeviceRadixSort (onesweep) + cub::DeviceScan -- library plumbing, like cuBLAS
  // for the towers.  RS_SORT=own selects the hand-written LSD radix sort and prefix sums of sort.cu: bit-identical
  // results (tests/test_kernels_gpu.py), but more and smaller launches, which measured 4 % slower on the whole C2 step
  // and 17 % on C5, so it is not the default.  head / segidx1 are free until the sort ends (its scratch).
  // The segment / chunk head flags are never stored on the cub path: the scans read them through transform iterators and
  // the later kernels recompute them (14 launches per dedup instead of 20 -- the small-batch configs are launch bound).
  const bool use_cub = !(getenv("RS_SORT") && !strcmp(getenv("RS_SORT"), "own"));
  int32_t *sort_hist = (int32_t *)(w + L.sort_hist), *scan_ws = (int32_t *)(w + L.scan_ws);
  using Count = cub::CountingInputIterator<int32_t>;
  if (use_cub) {
    RS_CUDA(cub::DeviceRadixSort::SortPairs(cub_ws, cub_bytes, keys_in, seg->sorted_key, pos_in, seg->sorted_pos, (int)n, 0, end_bit, st));
    cub::TransformInputIterator<int32_t, HeadOp, Count> heads(Count(0), HeadOp{seg->sorted_key, nvp, n});
    RS_CUDA(cub::DeviceScan::InclusiveSum(cub_ws, cub_bytes, heads, segidx1, (int)n, st));
  } else {
    int rc = rs::radix_sort_pairs(keys_in, pos_in, seg->sorted_key, seg->sorted_pos, (uint32_t *)head, segidx1, sort_hist, n, end_bit, st);
    if (rc) return rc;
    head_flags_kernel<<<blocks, 256, 0, st>>>(seg->sorted_key, n, head, nvp);
    RS_CHECK_LAUNCH();
    rc = rs::inclusive_sum_i32(head, segidx1, n, scan_ws, st);
    if (rc) return rc;
  }
  seg_scatter_kernel<<<blocks, 256, 0, st>>>(seg->sorted_key, seg->sorted_pos, segidx1, n, seg->uniq, seg->seg_start,
                                             seg->inverse, seg->n_uniq, nvp);
  RS_CHECK_LAUNCH();
  if (use_cub) {
    cub::TransformInputIterator<int32_t, ChunkHeadOp, Count> cheads(Count(0), ChunkHeadOp{segidx1, seg->seg_start, nvp, n});
    RS_CUDA(cub::DeviceScan::InclusiveSum(cub_ws, cub_bytes, cheads, chunkidx1, (int)n, st));
  } else {
    chunk_flags_kernel<<<blocks, 256, 0, st>>>(segidx1, seg->seg_start, n, chead, nvp);
    RS_CHECK_LAUNCH();
    int rc = rs::inclusive_sum_i32(chead, chunkidx1, n, scan_ws, st);
    if (rc) return rc;
  }
  chunk_scatter_kernel<<<blocks, 256, 0, st>>>(segidx1, seg->seg_start, chunkidx1, n, seg->chunk_start, seg->chunk_seg,
                                               seg->seg_first_chunk, seg->n_chunks, seg->counts, nvp);
  RS_CHECK_LAUNCH();
  const int nunits = (int)(n / RS_UNIT + 1);
  dedup_finish_kernel<<<blocks, 256, 0, st>>>(seg->sorted_pos, segidx1, chunkidx1, seg->seg_start, seg->chunk_start, seg->chunk_seg,
                                              seg->seg_first_chunk, seg->uniq, n, nunits, (int4 *)seg->lookup_desc, seg->unit_start,
                                              seg->n_uniq, seg->multi_seg, seg->n_multi, nvp);
  RS_CHECK_LAUNCH();
  return RS_OK;
}

RS_API int rs_segments_relabel(const rs_segments *seg, int64_t n, void *stream) {
  RS_CHECK_ARG(seg && seg->lookup_desc && seg->inverse && seg->uniq && seg->n_uniq, RS_E_ARG, "rs_segments_relabel: incomplete segments");
  if (n <= 0) return RS_OK;
  relabel_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((int4 *)seg->lookup_desc, seg->inverse, seg->uniq,
                                                                                seg->n_uniq, n);
  RS_CHECK_LAUNCH();
  return RS_OK;
}

// =================================================================== segment reduce + update
namespace {

using rs::partial_slot;

template <int VEC>
struct Vec;
template <>
struct Vec<4> {
  using T = float4;
  static __device__ __forceinline__ T zero() { return rs::f4_zero(); }
  static __device__ __forceinline__ T ld(const float *p) { return rs::ldg_f4(p); }
  static __device__ __forceinline__ T ldnc(const float *p) { return rs::ldg_nc_f4(p); }
  static __device__ __forceinline__ void st(float *p, T v) { rs::stg_f4(p, v); }
  static __device__ __forceinline__ T add(T a, T b) { return rs::f4_add(a, b); }
  static __device__ __forceinline__ T mul(T a, T b) { return rs::f4_mul(a, b); }
  static __device__ __forceinline__ T scale(T a, float s) { return rs::f4_scale(a, s); }
};
template <>
struct Vec<1> {
  using T = float;
  static __device__ __forceinline__ T zero() { return 0.f; }
  static __device__ __forceinline__ T ld(const float *p) { return *p; }
  static __device__ __forceinline__ T ldnc(const float *p) { return __ldg(p); }
  static __device__ __forceinline__ void st(float *p, T v) { *p = v; }
  static __device__ __forceinline__ T add(T a, T b) { return a + b; }
  static __device__ __forceinline__ T mul(T a, T b) { return a * b; }
  static __device__ __forceinline__ T scale(T a, float s) { return a * s; }
};

template <int VEC, int MODE>
__device__ __forceinline__ void apply_row(const UpdParams &P, const int64_t *rtab, int64_t row, int e /* element (in VEC units) */,
                                          typename Vec<VEC>::T g) {
  using V = Vec<VEC>;
  int64_t off = (row * P.W) + (int64_t)e * VEC;
  if (MODE == RS_UPD_GRAD) {
    if (P.routes.n > 0) {
      float *d = rs::route_row(P.routes, rtab, row, P.W);
      if (d) V::st(d + (int64_t)e * VEC, g);
    } else
      V::st(P.dense_grad + off, g);
  } else if (MODE == RS_UPD_SGD) {
    typename V::T w = V::ld(P.table + off);
    V::st(P.table + off, upd_sgd(w, g, P));
  } else {
    float wv[VEC], mv[VEC], vv[VEC], gv[VEC];
    *reinterpret_cast<typename V::T *>(wv) = V::ld(P.table + off);
    *reinterpret_cast<typename V::T *>(mv) = V::ld(P.m + off);
    *reinterpret_cast<typename V::T *>(vv) = V::ld(P.v + off);
    *reinterpret_cast<typename V::T *>(gv) = g;
#pragma unroll
    for (int i = 0; i < VEC; ++i) adam1(wv[i], mv[i], vv[i], gv[i], P);
    V::st(P.table + off, *reinterpret_cast<typename V::T *>(wv));
    V::st(P.m + off, *reinterpret_cast<typename V::T *>(mv));
    V::st(P.v + off, *reinterpret_cast<typename V::T *>(vv));
  }
}

// One lane group (GS lanes, NA elements of VEC floats per lane) per chunk.  Lookups of the chunk are visited in
// sorted (= ascending position) order; loads for UNR lookups are issued before their adds so the dependent FADD
// chain does not serialise the memory latency.
template <int VEC, int GS, int NA, int MODE>
__global__ void __launch_bounds__(256, (NA == 1) ? 6 : ((NA <= 4) ? 4 : 1)) seg_chunk_kernel(const __grid_constant__ UpdParams P, int64_t n) {
  using V = Vec<VEC>;
  constexpr int GPB = 256 / GS;
  __shared__ int64_t rtab[rs::ROUTE_TAB];
  if (MODE == RS_UPD_GRAD && P.routes.n > 0) {
    rs::route_tab_load(rtab, P.routes);
    __syncthreads();
  }
  const int lane = threadIdx.x % GS;
  const int WV = P.W / VEC;
  const int nchunks = *P.n_chunks;
  const int64_t crot = (MODE == RS_UPD_GRAD && P.routes.n > 0) ? rs::route_rotation(P.routes, nchunks) : 0;
  for (int64_t c0 = (int64_t)blockIdx.x * GPB + threadIdx.x / GS; c0 < nchunks; c0 += (int64_t)gridDim.x * GPB) {
    const int64_t c = c0 + crot < nchunks ? c0 + crot : c0 + crot - nchunks;   // all-to-all schedule (see rs_routes.self)
    const int s0 = P.chunk_start[c], s1 = P.chunk_start[c + 1];
    const int g = P.chunk_seg[c];
    // everything that depends only on g is requested now, so it is in flight together with the gradient rows
    const bool single = (P.seg_first_chunk[g + 1] - P.seg_first_chunk[g]) == 1;
    const int64_t row = P.uniq[g];
    typename V::T acc[NA];
#pragma unroll
    for (int a = 0; a < NA; ++a) acc[a] = V::zero();
    constexpr int UNR = (NA <= 2) ? 4 : (NA <= 4 ? 2 : 1);
    for (int s = s0; s < s1; s += UNR) {
      typename V::T val[UNR][NA];
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        const bool live = s + u < s1;
        const int p = live ? P.sorted_pos[s + u] : 0;
        const int b = p / P.F;
#pragma unroll
        for (int a = 0; a < NA; ++a) {
          const int e = lane + a * GS;
          typename V::T x = V::zero();
          if (live && e < WV) {
            if (P.stash) {
              x = V::ldnc(P.stash + (int64_t)p * P.W + e * VEC);
              if (P.scale) {
                if (P.scale_width == 1)
                  x = V::scale(x, __ldg(P.scale + b));
                else
                  x = V::mul(x, V::ldnc(P.scale + (int64_t)b * P.scale_width + e * VEC));
              }
            }
            if (P.dense) x = V::add(x, V::ldnc(P.dense + (int64_t)p * P.W + e * VEC));
          }
          val[u][a] = x;
        }
      }
#pragma unroll
      for (int u = 0; u < UNR; ++u)
#pragma unroll
        for (int a = 0; a < NA; ++a) acc[a] = V::add(acc[a], val[u][a]);
    }
    if (single) {
#pragma unroll
      for (int a = 0; a < NA; ++a) {
        const int e = lane + a * GS;
        if (e < WV) apply_row<VEC, MODE>(P, rtab, row, e, acc[a]);
      }
    } else {
      float *dst = P.partial + (int64_t)partial_slot(s0, s1 - s0) * P.W;
#pragma unroll
      for (int a = 0; a < NA; ++a) {
        const int e = lane + a * GS;
        if (e < WV) V::st(dst + e * VEC, acc[a]);
      }
    }
  }
}

// One CTA per segment that has more than one chunk.  Its 256/GS lane groups each add a contiguous run of the chunk
// partials in chunk order (loads of four partials issued before their adds); group 0 then adds the group sums in
// group order and applies the update.  The association is a fixed function of the segment length -> deterministic,
// and the hottest row (tens of thousands of lookups) no longer serialises ~hundreds of dependent memory latencies.
template <int VEC, int GS, int NA, int MODE>
__global__ void __launch_bounds__(256) seg_combine_kernel(const __grid_constant__ UpdParams P, int64_t n) {
  using V = Vec<VEC>;
  constexpr int GPB = 256 / GS;
  extern __shared__ __align__(16) float s_grp[];  // [GPB][W]
  __shared__ int64_t rtab[rs::ROUTE_TAB];
  if (MODE == RS_UPD_GRAD && P.routes.n > 0) {
    rs::route_tab_load(rtab, P.routes);
    __syncthreads();
  }
  const int lane = threadIdx.x % GS, grp = threadIdx.x / GS;
  const int WV = P.W / VEC;
  const int nm = *P.n_multi;
  for (int64_t k = blockIdx.x; k < nm; k += gridDim.x) {
    const int g = P.multi_seg[k];
    const int c0 = P.seg_first_chunk[g], c1 = P.seg_first_chunk[g + 1];
    const int per = (c1 - c0 + GPB - 1) / GPB;
    const int lo = c0 + grp * per, hi = (lo + per < c1) ? lo + per : c1;
    typename V::T acc[NA];
#pragma unroll
    for (int a = 0; a < NA; ++a) acc[a] = V::zero();
    constexpr int UNR = (NA <= 2) ? 4 : (NA <= 4 ? 2 : 1);
    for (int c = lo; c < hi; c += UNR) {
      typename V::T val[UNR][NA];
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        const bool live = c + u < hi;
        const int s0 = live ? P.chunk_start[c + u] : 0, s1 = live ? P.chunk_start[c + u + 1] : 0;
        const float *src = P.partial + (int64_t)partial_slot(s0, s1 - s0) * P.W;
#pragma unroll
        for (int a = 0; a < NA; ++a) {
          const int e = lane + a * GS;
          val[u][a] = (live && e < WV) ? V::ld(src + e * VEC) : V::zero();
        }
      }
#pragma unroll
      for (int u = 0; u < UNR; ++u)
#pragma unroll
        for (int a = 0; a < NA; ++a)
          if (c + u < hi) acc[a] = V::add(acc[a], val[u][a]);
    }
#pragma unroll
    for (int a = 0; a < NA; ++a) {
      const int e = lane + a * GS;
      if (e < WV) V::st(s_grp + (size_t)grp * P.W + e * VEC, acc[a]);
    }
    __syncthreads();
    if (grp == 0) {
      const int used = (c1 - c0 + per - 1) / per;  // groups that had at least one chunk
#pragma unroll
      for (int a = 0; a < NA; ++a) {
        const int e = lane + a * GS;
        if (e < WV) {
          typename V::T t = V::ld(s_grp + e * VEC);
          for (int q = 1; q < used; ++q) t = V::add(t, V::ld(s_grp + (size_t)q * P.W + e * VEC));
          apply_row<VEC, MODE>(P, rtab, P.uniq[g], e, t);
        }
      }
    }
    __syncthreads();
  }
}

template <int VEC, int GS, int NA, int MODE>
int launch_update(const UpdParams &P, int64_t n, cudaStream_t st) {
  constexpr int GPB = 256 / GS;
  int64_t blocks64 = (n + GPB - 1) / GPB;
  int cap = rs::num_sms() * 64;
  int blocks = (int)(blocks64 < cap ? blocks64 : cap);
  if (P.combine_only) {
    // the chunk pass was done by another kernel (ffm_train.cu) that left the partials of the multi-chunk segments in P.partial
  } else if (P.use_stream) {
    int rc = rs::launch_seg_stream(P, n, MODE, st);   // chunk pass as a TMA-fed streaming kernel (segment_stream.cu)
    if (rc) return rc;
  } else {
    seg_chunk_kernel<VEC, GS, NA, MODE><<<blocks, 256, 0, st>>>(P, n);
  }
  RS_CHECK_LAUNCH();
  // a multi-chunk segment has > RS_CHUNK lookups, so there are at most n / RS_CHUNK of them
  int64_t cblocks64 = n / RS_CHUNK + 1;
  int cblocks = (int)(cblocks64 < rs::num_sms() * 8 ? cblocks64 : rs::num_sms() * 8);
  const size_t csmem = (size_t)GPB * P.W * 4;
  if (csmem > 48 * 1024)
    RS_CUDA(cudaFuncSetAttribute(seg_combine_kernel<VEC, GS, NA, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)csmem));
  seg_combine_kernel<VEC, GS, NA, MODE><<<cblocks, 256, csmem, st>>>(P, n);
  RS_CHECK_LAUNCH();
  return RS_OK;
}

template <int VEC, int GS, int NA>
int launch_mode(const UpdParams &P, int mode, int64_t n, cudaStream_t st) {
  switch (mode) {
    case RS_UPD_GRAD: return launch_update<VEC, GS, NA, RS_UPD_GRAD>(P, n, st);
    case RS_UPD_SGD: return launch_update<VEC, GS, NA, RS_UPD_SGD>(P, n, st);
    case RS_UPD_ADAM: return launch_update<VEC, GS, NA, RS_UPD_ADAM>(P, n, st);
  }
  rs::set_error("rs_segment_update: bad mode %d", mode);
  return RS_E_ARG;
}

}  // namespace

namespace rs {

void set_opt_scalars(const rs_update *u, UpdParams &P) {
  P.lr = u->lr;
  P.wd = u->wd;
  P.beta1 = u->beta1;
  P.beta2 = u->beta2;
  P.eps = u->eps;
  double bc1 = 1.0 - pow((double)u->beta1, (double)u->step);
  double bc2 = 1.0 - pow((double)u->beta2, (double)u->step);
  P.step_size = (float)((double)u->lr / (bc1 > 0 ? bc1 : 1.0));
  P.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2 > 0 ? bc2 : 1.0));
}

int make_upd_params(const rs_segments *seg, int64_t n, const rs_update *u, UpdParams &P) {
  RS_CHECK_ARG((int64_t)(2 * (n / RS_CHUNK + 2)) * u->width <= seg->partial_floats, RS_E_WORKSPACE,
               "rs_segment_update: dedup workspace was sized for a narrower row (need %lld floats of partials, have %lld)",
               (long long)((int64_t)(2 * (n / RS_CHUNK + 2)) * u->width), (long long)seg->partial_floats);
  P.sorted_pos = seg->sorted_pos;
  P.seg_start = seg->seg_start;
  P.seg_first_chunk = seg->seg_first_chunk;
  P.chunk_start = seg->chunk_start;
  P.chunk_seg = seg->chunk_seg;
  P.n_uniq = seg->n_uniq;
  P.n_chunks = seg->n_chunks;
  P.multi_seg = seg->multi_seg;
  P.n_multi = seg->n_multi;
  P.lookup_desc = (const int4 *)seg->lookup_desc;
  P.work_counter = seg->work_counter;
  P.unit_start = seg->unit_start;
  P.scale_sorted = seg->scale_sorted;
  P.uniq = seg->uniq;
  P.partial = seg->partial;
  P.stash = u->stash;
  P.scale = u->scale;
  P.dense = u->dense;
  P.table = u->table;
  P.m = u->m;
  P.v = u->v;
  P.dense_grad = u->dense_grad;
  P.routes.n = 0;
  P.routes.dyn_start = P.routes.dyn_row0 = nullptr;
  P.routes.cap_rows = 0;
  P.routes.self = -1;
  if (u->mode == RS_UPD_GRAD && u->grad_routes) {
    int rc = rs::fill_routes(P.routes, u->grad_routes, "rs_segment_update");
    if (rc) return rc;
  }
  P.W = u->width;
  P.F = u->F;
  P.scale_width = u->scale_width;
  set_opt_scalars(u, P);
  P.use_stream = 0;
  P.combine_only = 0;
  P.half_sm = u->half_sm;
  return RS_OK;
}

// chunk pass + combine pass (or the combine pass alone when P.combine_only) for rows of P.W floats
int dispatch_update(const UpdParams &P, int mode, int64_t n, cudaStream_t st) {
  const int W = P.W;
  if (W % 4 == 0) {
    const int wv = W / 4;
    if (wv <= 1) return launch_mode<4, 1, 1>(P, mode, n, st);
    if (wv <= 2) return launch_mode<4, 2, 1>(P, mode, n, st);
    if (wv <= 4) return launch_mode<4, 4, 1>(P, mode, n, st);
    if (wv <= 8) return launch_mode<4, 8, 1>(P, mode, n, st);
    if (wv <= 16) return launch_mode<4, 16, 1>(P, mode, n, st);
    if (wv <= 32) return launch_mode<4, 32, 1>(P, mode, n, st);
    if (wv <= 64) return launch_mode<4, 32, 2>(P, mode, n, st);
    if (wv <= 128) return launch_mode<4, 32, 4>(P, mode, n, st);
    if (wv <= 256) return launch_mode<4, 32, 8>(P, mode, n, st);
    return launch_mode<4, 32, 16>(P, mode, n, st);
  }
  if (W == 1) return launch_mode<1, 1, 1>(P, mode, n, st);
  if (W <= 32) return launch_mode<1, 32, 1>(P, mode, n, st);
  if (W <= 128) return launch_mode<1, 32, 4>(P, mode, n, st);
  if (W <= 512) return launch_mode<1, 32, 16>(P, mode, n, st);
  rs::set_error("rs_segment_update: width %d not a multiple of 4 and > 512", W);
  return RS_E_UNSUPPORTED;
}

}  // namespace rs

RS_API int rs_segment_update(const rs_segments *seg, int64_t n, const rs_update *u, void *stream) {
  RS_CHECK_ARG(seg && u, RS_E_ARG, "rs_segment_update: null argument");
  RS_CHECK_ARG(n > 0 && n < (1ll << 31), RS_E_SHAPE, "rs_segment_update: bad n");
  RS_CHECK_ARG(u->width >= 1 && u->width <= 2048 && u->F >= 1 && n % u->F == 0, RS_E_SHAPE, "rs_segment_update: bad width/F");
  RS_CHECK_ARG(u->stash || u->dense, RS_E_ARG, "rs_segment_update: need stash and/or dense gradient source");
  RS_CHECK_ARG(!u->scale || (u->stash && (u->scale_width == 1 || u->scale_width == u->width)), RS_E_ARG,
               "rs_segment_update: scale needs stash and scale_width in {1,width}");
  if (u->mode == RS_UPD_GRAD) RS_CHECK_ARG(u->dense_grad || u->grad_routes, RS_E_ARG, "rs_segment_update: dense_grad is NULL");
  if (u->mode != RS_UPD_GRAD) RS_CHECK_ARG(u->table, RS_E_ARG, "rs_segment_update: table is NULL");
  if (u->mode == RS_UPD_ADAM) RS_CHECK_ARG(u->m && u->v && u->step >= 1, RS_E_ARG, "rs_segment_update: Adam needs m, v, step>=1");
  UpdParams P;
  int rc = rs::make_upd_params(seg, n, u, P);
  if (rc) return rc;
  const int W = u->width;
  // wide rows (>= 384 B) with one gradient source and at most a per-sample scalar scale take the TMA-fed streaming kernel;
  // at 256 B (DIN / MF item rows) the lane-group kernel is faster (0.11 vs 0.26 ms on the C4 batch: the streaming kernel is
  // bound by its per-row bulk-copy issue rate, not by bytes)
  P.use_stream = (W % 4 == 0 && W >= 96 && W <= 640 && !(u->stash && u->dense) && (!u->scale || u->scale_width == 1) &&
                  !getenv("RS_NO_STREAM")) ? 1 : 0;
  return rs::dispatch_update(P, u->mode, n, (cudaStream_t)stream);
}

// =================================================================== dense Adam sweep
__global__ void __launch_bounds__(256) adam_dense_kernel(float *__restrict__ p, const float *__restrict__ g, float *__restrict__ m,
                                                        float *__restrict__ v, int64_t numel, float wd, float beta1, float beta2, float eps,
                                                        float step_size, float inv_sqrt_bc2) {
  UpdParams P;
  P.wd = wd;
  P.beta1 = beta1;
  P.beta2 = beta2;
  P.eps = eps;
  P.step_size = step_size;
  P.inv_sqrt_bc2 = inv_sqrt_bc2;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < numel; i += (int64_t)gridDim.x * blockDim.x) {
    float w = p[i], mm = m[i], vv = v[i];
    adam1(w, mm, vv, g[i], P);
    p[i] = w;
    m[i] = mm;
    v[i] = vv;
  }
}

RS_API int rs_adam_dense(float *p, const float *g, float *m, float *v, int64_t numel, float lr, float wd, float beta1, float beta2,
                         float eps, int32_t step, void *stream) {
  RS_CHECK_ARG(p && g && m && v && step >= 1, RS_E_ARG, "rs_adam_dense: bad argument");
  if (numel == 0) return RS_OK;
  double bc1 = 1.0 - pow((double)beta1, (double)step);
  double bc2 = 1.0 - pow((double)beta2, (double)step);
  int64_t blocks64 = (numel + 255) / 256;
  int cap = rs::num_sms() * 16;
  int blocks = (int)(blocks64 < cap ? blocks64 : cap);
  adam_dense_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(p, g, m, v, numel, wd, beta1, beta2, eps, (float)((double)lr / bc1),
                                                              (float)(1.0 / sqrt(bc2)));
  RS_CHECK_LAUNCH();
  return RS_OK;
}
