// Row-sharded tables: the exchange plan of a step, kept entirely on the device (no reference counterpart; SURVEY.md 8e).
//
// Global row g lives on rank g % N at local index g / N.  A requester's distinct rows arrive here already sorted
// owner-major (rs_dedup_sort_ex with shard_world), so the rows wanted from owner o are the contiguous range
// [bounds[o], bounds[o+1]) of `uniq`.  Counts, offsets and request lists are written straight into the owners' symmetric
// (peer-mapped) `req` / `ctl` buffers over NVLink; after one cross-rank barrier every owner knows what to serve and
// where each requester's gradients will land.  Nothing is read back by the host, so the whole sharded train step is a
// fixed launch sequence (CUDA-graph capturable).
//
// rs_shard_serve is the "rows" all-to-all fused into the owner's gather: for wide rows (FFM, 1664 B) each warp runs a
// TMA pipeline -- cp.async.bulk global->shared of up to SERVE_C table rows into a stage, then ONE cp.async.bulk
// shared->global of the whole stage into the requester's block (contiguous there), so the SM issues two bulk copies per
// 16 rows and the payload never touches registers.  Narrow rows (FM, 64 B) use 128-bit loads/stores.
#include <stdlib.h>
#include <string.h>

#include "segment.cuh"

namespace {

struct ShardDev {
  int world, rank;
  int64_t R, cap_req, cap_recv;
  int32_t *req[RS_MAX_RANKS];
  int64_t *ctl[RS_MAX_RANKS];
  int n_direct;
  int64_t direct_lo[RS_MAX_DIRECT], direct_hi[RS_MAX_DIRECT];
};

int fill_shard(ShardDev &D, const rs_shard *S, const char *who) {
  RS_CHECK_ARG(S && S->world >= 1 && S->world <= RS_MAX_RANKS && S->rank >= 0 && S->rank < S->world, RS_E_ARG, "%s: bad world/rank", who);
  RS_CHECK_ARG(S->rows_per_rank > 0 && S->cap_req > 0 && S->cap_recv > 0, RS_E_ARG, "%s: bad capacities", who);
  D.world = S->world, D.rank = S->rank, D.R = S->rows_per_rank, D.cap_req = S->cap_req, D.cap_recv = S->cap_recv;
  for (int k = 0; k < S->world; ++k) {
    RS_CHECK_ARG(S->req[k] && S->ctl[k], RS_E_ARG, "%s: null peer buffer for rank %d", who, k);
    D.req[k] = S->req[k];
    D.ctl[k] = S->ctl[k];
  }
  RS_CHECK_ARG(S->n_direct >= 0 && S->n_direct <= RS_MAX_DIRECT, RS_E_ARG, "%s: at most %d direct ranges", who, RS_MAX_DIRECT);
  RS_CHECK_ARG(S->n_direct == 0 || S->rows_per_rank < (1ll << 31), RS_E_SHAPE, "%s: direct ranges need rows_per_rank < 2^31", who);
  D.n_direct = S->n_direct;
  for (int k = 0; k < S->n_direct; ++k) D.direct_lo[k] = S->direct_lo[k], D.direct_hi[k] = S->direct_hi[k];
  return RS_OK;
}

// first index j in [0, n) with a[j] >= key
__device__ __forceinline__ int64_t lower_bound(const int64_t *__restrict__ a, int64_t n, int64_t key) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (a[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// ------------------------------------------------------------------ requester: post the request lists
__global__ void __launch_bounds__(256) shard_post_kernel(const __grid_constant__ ShardDev S, const int64_t *__restrict__ uniq,
                                                        const int32_t *__restrict__ n_uniq) {
  __shared__ int64_t bounds[RS_MAX_RANKS + 1];
  const int64_t nu = *n_uniq;
  if (threadIdx.x <= S.world) bounds[threadIdx.x] = lower_bound(uniq, nu, (int64_t)threadIdx.x * S.R);
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x <= S.world) {
    const int o = threadIdx.x;
    S.ctl[S.rank][RS_CTL_SEND_START + o] = bounds[o];
    if (o < S.world) {
      S.ctl[o][RS_CTL_CNT_IN + S.rank] = bounds[o + 1] - bounds[o];   // rows I want from owner o
      S.ctl[o][RS_CTL_BLK0_IN + S.rank] = bounds[o];                  // ... and where they belong inside my block
    }
  }
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nu; j += (int64_t)gridDim.x * blockDim.x) {
    const int64_t key = uniq[j];
    const int o = (int)(key / S.R);
    const int64_t l = key - (int64_t)o * S.R;
    uint32_t e = (uint32_t)l;
    if (S.n_direct > 0) {          // flag rows of the direct ranges: the owner will not copy them (bit 31)
      const int64_t g = l * S.world + o;
      for (int k = 0; k < S.n_direct; ++k)
        if (g >= S.direct_lo[k] && g < S.direct_hi[k]) e |= 0x80000000u;
    }
    S.req[o][(int64_t)S.rank * S.cap_req + (j - bounds[o])] = (int32_t)e;
  }
}

// ------------------------------------------------------------------ owner: prefix of the counts + compact receive list
__global__ void __launch_bounds__(256) shard_collect_kernel(const __grid_constant__ ShardDev S, int64_t *__restrict__ recv_local,
                                                           uint8_t *__restrict__ recv_skip, int32_t *__restrict__ m_total,
                                                           int32_t *status) {
  __shared__ int64_t start[RS_MAX_RANKS + 1];
  int64_t *ctl = S.ctl[S.rank];
  if (threadIdx.x == 0) {
    int64_t acc = 0;
    for (int r = 0; r < S.world; ++r) {
      start[r] = acc < S.cap_recv ? acc : S.cap_recv;
      acc += ctl[RS_CTL_CNT_IN + r];
    }
    if (acc > S.cap_recv) {      // more rows than the receive buffers hold: flagged, the surplus is dropped everywhere
      if (status && blockIdx.x == 0) atomicOr(status, 16);
      acc = S.cap_recv;
    }
    start[S.world] = acc;
  }
  __syncthreads();
  if (blockIdx.x == 0) {
    if (threadIdx.x <= S.world) ctl[RS_CTL_RECV_START + threadIdx.x] = start[threadIdx.x];
    if (threadIdx.x < S.world) S.ctl[threadIdx.x][RS_CTL_G0_IN + S.rank] = start[threadIdx.x];   // requester r pushes its gradients here
    if (threadIdx.x == 0) {
      ctl[RS_CTL_M_TOTAL] = start[S.world];
      *m_total = (int32_t)start[S.world];
    }
  }
  const int64_t m = start[S.world];
  const int32_t *req = S.req[S.rank];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    int r = 0;
    while (r + 1 < S.world && i >= start[r + 1]) ++r;
    const uint32_t e = (uint32_t)req[(int64_t)r * S.cap_req + (i - start[r])];
    recv_local[i] = (int64_t)(e & 0x7fffffffu);
    if (recv_skip) recv_skip[i] = (uint8_t)(e >> 31);
  }
}

// ------------------------------------------------------------------ owner: serve the rows
struct Blocks {
  float *base[RS_MAX_RANKS];
};

// generic 128-bit path (any width that is a multiple of 4 floats): one 16-byte piece per thread iteration, four in flight
__global__ void __launch_bounds__(256) shard_serve_kernel(const __grid_constant__ ShardDev S, const float *__restrict__ table, int64_t rows,
                                                         int wv, const int64_t *__restrict__ recv_local,
                                                         const uint8_t *__restrict__ skip, const __grid_constant__ Blocks B,
                                                         int64_t cap_block, int32_t *status) {
  __shared__ int64_t start[RS_MAX_RANKS + 1], blk0[RS_MAX_RANKS];
  const int64_t *ctl = S.ctl[S.rank];
  if (threadIdx.x <= S.world) start[threadIdx.x] = ctl[RS_CTL_RECV_START + threadIdx.x];
  if (threadIdx.x < S.world) blk0[threadIdx.x] = ctl[RS_CTL_BLK0_IN + threadIdx.x];
  __syncthreads();
  const int64_t total = start[S.world] * wv;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  // all-to-all schedule: owner o serves requester o+1 first, then o+2, ... so the owners never gang up on one receiver
  const int64_t rot = start[(S.rank + 1) % S.world] * wv;
  for (int64_t e0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e0 < total; e0 += 4 * stride) {
    float4 val[4];
    float *dst[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t ev = e0 + u * stride;
      const int64_t e = ev + rot < total ? ev + rot : ev + rot - total;
      dst[u] = nullptr;
      if (ev < total && !(skip && skip[e / wv])) {
        const int64_t i = e / wv;
        const int v = (int)(e - i * wv);
        int r = 0;
        while (r + 1 < S.world && i >= start[r + 1]) ++r;
        const int64_t id = rs::clamp_id(recv_local[i], rows, status);
        const int64_t drow = blk0[r] + (i - start[r]);
        val[u] = rs::ldg_nc_f4(table + (id * wv + v) * 4);
        if (drow < cap_block) dst[u] = B.base[r] + (drow * wv + v) * 4;
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (dst[u]) rs::stg_f4(dst[u], val[u]);
  }
}

// TMA path.  Every warp owns SERVE_NST stages of SERVE_C rows.  Work item = up to SERVE_C consecutive rows of ONE
// requester's list (they are consecutive in its block, so a stage leaves in a single bulk store).
constexpr int SERVE_C = 16, SERVE_NST = 2, SERVE_WARPS = 4;

__global__ void __launch_bounds__(SERVE_WARPS * 32, 1) shard_serve_tma_kernel(const __grid_constant__ ShardDev S, const float *__restrict__ table,
                                                                             int64_t rows, int W, const int64_t *__restrict__ recv_local,
                                                                             const uint8_t *__restrict__ skip,
                                                                             const __grid_constant__ Blocks B, int64_t cap_block,
                                                                             int32_t *status) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint64_t full_bar[SERVE_WARPS][SERVE_NST];
  __shared__ int64_t start[RS_MAX_RANKS + 1], blk0[RS_MAX_RANKS], cstart[RS_MAX_RANKS + 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t row_bytes = (uint32_t)W * 4u;
  const int64_t *ctl = S.ctl[S.rank];
  if (threadIdx.x <= S.world) start[threadIdx.x] = ctl[RS_CTL_RECV_START + threadIdx.x];
  if (threadIdx.x < S.world) blk0[threadIdx.x] = ctl[RS_CTL_BLK0_IN + threadIdx.x];
  if (threadIdx.x < SERVE_WARPS * SERVE_NST) rs::mbar_init(&full_bar[threadIdx.x / SERVE_NST][threadIdx.x % SERVE_NST], 1);
  __syncthreads();
  if (threadIdx.x == 0) {
    // chunk numbering follows the all-to-all schedule: position i of the walk serves requester (rank + 1 + i) % world, so
    // the owners never gang up on one receiver's NVLink ingress
    int64_t acc = 0;
    for (int i = 0; i < S.world; ++i) {
      const int r = (S.rank + 1 + i) % S.world;
      cstart[i] = acc;
      acc += (start[r + 1] - start[r] + SERVE_C - 1) / SERVE_C;
    }
    cstart[S.world] = acc;
    rs::mbar_fence_init();
  }
  __syncthreads();
  const int64_t nchunks = cstart[S.world];
  float *ring = reinterpret_cast<float *>(smem_raw) + (size_t)warp * SERVE_NST * SERVE_C * W;
  const int64_t gw = (int64_t)blockIdx.x * SERVE_WARPS + warp, nw = (int64_t)gridDim.x * SERVE_WARPS;
  const int64_t mine = gw < nchunks ? (nchunks - gw + nw - 1) / nw : 0;   // chunks gw, gw + nw, ...

  // chunk k of this warp -> (first compact row, row count, destination)
  auto describe = [&](int64_t k, int64_t &i0, int &cnt, float *&dst) {
    const int64_t c = gw + k * nw;
    int i = 0;
    while (i + 1 < S.world && c >= cstart[i + 1]) ++i;
    const int r = (S.rank + 1 + i) % S.world;
    i0 = start[r] + (c - cstart[i]) * SERVE_C;
    const int64_t left = start[r + 1] - i0;
    cnt = (int)(left < SERVE_C ? left : SERVE_C);
    const int64_t drow = blk0[r] + (i0 - start[r]);
    if (drow + cnt > cap_block) cnt = drow < cap_block ? (int)(cap_block - drow) : 0;
    dst = B.base[r] + drow * W;
  };

  // iteration k: [stage k % NST is free once the store of chunk k - NST has read it] -> loads of chunk k ->
  // [wait for the loads of chunk k - 1] -> store of chunk k - 1.  The store of chunk k - NST was committed NST - 2
  // groups ago, so at most NST - 2 newer groups may still be reading.  live[st]: rows of the chunk that are copied at all
  // (rows of a "direct" range are skipped); a fully live chunk leaves in one bulk store, a mixed one in one store per run.
  uint32_t live[SERVE_NST];
  for (int64_t k = 0; k <= mine; ++k) {
    if (k < mine) {
      const int st = (int)(k % SERVE_NST);
      if (lane == 0) rs::bulk_wait_read<SERVE_NST - 2>();
      __syncwarp();
      int64_t i0;
      int cnt;
      float *dst;
      describe(k, i0, cnt, dst);
      const bool on = lane < cnt && !(skip && skip[i0 + lane]);
      live[st] = __ballot_sync(0xffffffffu, on);
      if (lane == 0) rs::mbar_arrive_expect_tx(&full_bar[warp][st], row_bytes * (uint32_t)__popc(live[st]));
      __syncwarp();
      if (on) {
        const int64_t id = rs::clamp_id(recv_local[i0 + lane], rows, status);
        rs::bulk_g2s(ring + ((size_t)st * SERVE_C + lane) * W, table + id * W, row_bytes, &full_bar[warp][st]);
      }
    }
    const int64_t j = k - 1;
    if (j >= 0 && lane == 0) {
      const int st = (int)(j % SERVE_NST);
      int64_t i0;
      int cnt;
      float *dst;
      describe(j, i0, cnt, dst);
      rs::mbar_wait(&full_bar[warp][st], (uint32_t)(j / SERVE_NST) & 1u);
      uint32_t m = live[st];
      while (m) {                                   // maximal runs of copied rows (one run in the common case)
        const int a = __ffs(m) - 1;
        const uint32_t rest = ~(m >> a);
        const int len = rest ? __ffs(rest) - 1 : 32 - a;
        rs::bulk_s2g(dst + (size_t)a * W, ring + ((size_t)st * SERVE_C + a) * W, row_bytes * (uint32_t)len);
        m = (len + a >= 32) ? 0u : (m >> (a + len)) << (a + len);
      }
      rs::bulk_commit();
    }
    __syncwarp();
  }
  if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ------------------------------------------------------------------ replicated small tables: all-reduce fused with the SGD step
// Every rank holds the same copy `w` of the small tables and its own dense gradient `g` (both in symmetric memory).  Rank r
// owns the r-th slice of the elements: it adds the N gradient slices in rank order (peer loads over NVLink), applies the
// SGD step to its own copy's values and stores the new values into EVERY rank's copy (peer stores).  One kernel is the
// reduce-scatter, the optimizer step and the all-gather; each element is computed once, so the replicas stay bit-identical.
struct Replicas {
  float *w[RS_MAX_RANKS];
  const float *g[RS_MAX_RANKS];
};

__global__ void __launch_bounds__(256) replica_sgd_kernel(const __grid_constant__ Replicas R, int world, int rank, int64_t lo4, int64_t hi4,
                                                         float lr, float wd) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = lo4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi4; i += stride) {
    float4 acc = rs::f4_zero();
    for (int r0 = 0; r0 < world; r0 += 8) {      // eight peer loads in flight, added in rank order
      float4 v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = (r0 + k < world) ? rs::ldg_f4(R.g[r0 + k] + i * 4) : rs::f4_zero();
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (r0 + k < world) acc = rs::f4_add(acc, v[k]);
    }
    const float4 w = rs::ldg_f4(R.w[rank] + i * 4);
    const float4 n = make_float4(w.x - lr * (acc.x + wd * w.x), w.y - lr * (acc.y + wd * w.y), w.z - lr * (acc.z + wd * w.z),
                                 w.w - lr * (acc.w + wd * w.w));
    for (int r = 0; r < world; ++r) rs::stg_f4(R.w[(rank + r) % world] + i * 4, n);
  }
}

// ------------------------------------------------------------------ replicated small tables: lazy row update (SGD / Adam)
// Same slicing, rank-ordered sum and store into every replica as replica_sgd_kernel, but only rows that some rank's batch
// touched move (touched[r][row] != 0 for some r) -- the single-GPU row update is lazy, and an untouched row must keep its
// bits under Adam (m != 0 keeps moving w) and weight decay.  The flags decide, not the gradient: a touched row whose summed
// gradient is exactly zero still steps.  The arithmetic is the row-update kernels' (upd_sgd / adam1, segment.cuh).
// Adam's m and v are not replicated: only this rank's slice exists, indexed from lo4.
struct Flags {
  const uint8_t *t[RS_MAX_RANKS];
};

template <int MODE>
__global__ void __launch_bounds__(256) replica_update_kernel(const __grid_constant__ Replicas R, const __grid_constant__ Flags T, int world,
                                                            int rank, int64_t lo4, int64_t hi4, int wv, float *__restrict__ m_slice,
                                                            float *__restrict__ v_slice, float lr, float wd, float beta1, float beta2,
                                                            float eps, float step_size, float inv_sqrt_bc2) {
  rs::UpdParams P;
  P.lr = lr;
  P.wd = wd;
  P.beta1 = beta1;
  P.beta2 = beta2;
  P.eps = eps;
  P.step_size = step_size;
  P.inv_sqrt_bc2 = inv_sqrt_bc2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = lo4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi4; i += stride) {
    // width % 4 == 0: a float4 never straddles two rows (32-bit division where it fits: the 64-bit one is emulated)
    const int64_t row = hi4 <= 0xffffffffll ? (int64_t)((uint32_t)i / (uint32_t)wv) : i / wv;
    uint32_t hit = 0;
    for (int r0 = 0; r0 < world; r0 += 8) {
      uint32_t f[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) f[k] = (r0 + k < world) ? T.t[r0 + k][row] : 0u;
#pragma unroll
      for (int k = 0; k < 8; ++k) hit |= f[k];
    }
    if (!hit) continue;
    float4 acc = rs::f4_zero();
    for (int r0 = 0; r0 < world; r0 += 8) {      // replica_sgd_kernel's sum: eight peer loads in flight, rank order
      float4 v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = (r0 + k < world) ? rs::ldg_f4(R.g[r0 + k] + i * 4) : rs::f4_zero();
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (r0 + k < world) acc = rs::f4_add(acc, v[k]);
    }
    float4 w = rs::ldg_f4(R.w[rank] + i * 4);
    if (MODE == RS_UPD_SGD) {
      w = rs::upd_sgd(w, acc, P);
    } else {
      float *mp = m_slice + (i - lo4) * 4, *vp = v_slice + (i - lo4) * 4;
      float4 m = rs::ldg_f4(mp), v = rs::ldg_f4(vp);
      rs::adam1(w.x, m.x, v.x, acc.x, P);
      rs::adam1(w.y, m.y, v.y, acc.y, P);
      rs::adam1(w.z, m.z, v.z, acc.z, P);
      rs::adam1(w.w, m.w, v.w, acc.w, P);
      rs::stg_f4(mp, m);
      rs::stg_f4(vp, v);
    }
    for (int r = 0; r < world; ++r) rs::stg_f4(R.w[(rank + r) % world] + i * 4, w);
  }
}

__global__ void __launch_bounds__(256) mark_rows_kernel(const int64_t *__restrict__ uniq, const int32_t *__restrict__ n_uniq,
                                                       uint8_t *__restrict__ touched, int64_t rows, int32_t *status) {
  const int64_t nu = *n_uniq;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nu; j += (int64_t)gridDim.x * blockDim.x)
    touched[rs::clamp_id(uniq[j], rows, status)] = 1;
}

// rank `rank`'s float4 slice [lo4, hi4) of n4: per = ceil(n4 / world)
void replica_slice(int64_t n4, int world, int rank, int64_t &lo4, int64_t &hi4) {
  const int64_t per = (n4 + world - 1) / world;
  lo4 = per * rank < n4 ? per * rank : n4;
  hi4 = lo4 + per < n4 ? lo4 + per : n4;
}

}  // namespace

RS_API int rs_replica_sgd(float *const *w, const float *const *g, int64_t numel, int32_t world, int32_t rank, float lr, float wd,
                          void *stream) {
  RS_CHECK_ARG(w && g && world >= 1 && world <= RS_MAX_RANKS && rank >= 0 && rank < world, RS_E_ARG, "rs_replica_sgd: bad argument");
  RS_CHECK_ARG(numel >= 0 && numel % 4 == 0, RS_E_SHAPE, "rs_replica_sgd: numel must be a multiple of 4");
  Replicas R;
  for (int k = 0; k < world; ++k) {
    RS_CHECK_ARG(w[k] && g[k], RS_E_ARG, "rs_replica_sgd: null buffer for rank %d", k);
    R.w[k] = w[k];
    R.g[k] = g[k];
  }
  int64_t lo4, hi4;
  replica_slice(numel / 4, world, rank, lo4, hi4);
  if (hi4 <= lo4) return RS_OK;
  int64_t blocks = (hi4 - lo4 + 255) / 256;
  const int cap = rs::num_sms() * 8;
  replica_sgd_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, (cudaStream_t)stream>>>(R, world, rank, lo4, hi4, lr, wd);
  RS_CHECK_LAUNCH();
  return RS_OK;
}

RS_API int rs_mark_rows(const rs_segments *seg, int64_t n, uint8_t *touched, int64_t rows, int32_t *status, void *stream) {
  RS_CHECK_ARG(seg && seg->uniq && seg->n_uniq && touched, RS_E_ARG, "rs_mark_rows: null argument");
  RS_CHECK_ARG(n > 0 && rows > 0, RS_E_SHAPE, "rs_mark_rows: bad n / rows");
  int64_t blocks = (n + 255) / 256;
  const int cap = rs::num_sms() * 8;
  mark_rows_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, (cudaStream_t)stream>>>(seg->uniq, seg->n_uniq, touched, rows, status);
  RS_CHECK_LAUNCH();
  return RS_OK;
}

RS_API int rs_replica_update(float *const *w, const float *const *g, const uint8_t *const *touched, int64_t numel, int32_t world,
                             int32_t rank, const rs_update *u, void *stream) {
  RS_CHECK_ARG(w && g && touched && u && world >= 1 && world <= RS_MAX_RANKS && rank >= 0 && rank < world, RS_E_ARG,
               "rs_replica_update: bad argument");
  RS_CHECK_ARG(u->mode == RS_UPD_SGD || u->mode == RS_UPD_ADAM, RS_E_UNSUPPORTED, "rs_replica_update: mode must be RS_UPD_SGD or RS_UPD_ADAM");
  RS_CHECK_ARG(u->width >= 4 && u->width % 4 == 0 && numel >= 0 && numel % u->width == 0, RS_E_SHAPE,
               "rs_replica_update: width must be a multiple of 4 that divides numel");
  if (u->mode == RS_UPD_ADAM) RS_CHECK_ARG(u->step >= 1, RS_E_ARG, "rs_replica_update: Adam needs step >= 1");
  Replicas R;
  Flags T;
  for (int k = 0; k < world; ++k) {
    RS_CHECK_ARG(w[k] && g[k] && touched[k], RS_E_ARG, "rs_replica_update: null buffer for rank %d", k);
    R.w[k] = w[k];
    R.g[k] = g[k];
    T.t[k] = touched[k];
  }
  int64_t lo4, hi4;
  replica_slice(numel / 4, world, rank, lo4, hi4);
  if (hi4 <= lo4) return RS_OK;
  if (u->mode == RS_UPD_ADAM) RS_CHECK_ARG(u->m && u->v, RS_E_ARG, "rs_replica_update: Adam needs this rank's m and v slices");
  rs::UpdParams P;
  rs::set_opt_scalars(u, P);
  int64_t blocks = (hi4 - lo4 + 255) / 256;
  const int cap = rs::num_sms() * 8;
  const int grid = (int)(blocks < cap ? blocks : cap);
  cudaStream_t st = (cudaStream_t)stream;
  if (u->mode == RS_UPD_SGD)
    replica_update_kernel<RS_UPD_SGD><<<grid, 256, 0, st>>>(R, T, world, rank, lo4, hi4, u->width / 4, nullptr, nullptr, P.lr, P.wd,
                                                            P.beta1, P.beta2, P.eps, P.step_size, P.inv_sqrt_bc2);
  else
    replica_update_kernel<RS_UPD_ADAM><<<grid, 256, 0, st>>>(R, T, world, rank, lo4, hi4, u->width / 4, u->m, u->v, P.lr, P.wd,
                                                             P.beta1, P.beta2, P.eps, P.step_size, P.inv_sqrt_bc2);
  RS_CHECK_LAUNCH();
  return RS_OK;
}

RS_API int rs_shard_post(const rs_shard *S, const rs_segments *seg, int64_t n, int32_t *status, void *stream) {
  ShardDev D;
  if (int rc = fill_shard(D, S, "rs_shard_post")) return rc;
  RS_CHECK_ARG(seg && seg->uniq && seg->n_uniq, RS_E_ARG, "rs_shard_post: incomplete segments");
  RS_CHECK_ARG(n > 0 && n <= S->cap_req, RS_E_SHAPE, "rs_shard_post: %lld lookups exceed the request-slot capacity %lld", (long long)n,
               (long long)S->cap_req);
  (void)status;
  int64_t blocks = (n + 255) / 256;
  const int cap = rs::num_sms() * 8;
  shard_post_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, (cudaStream_t)stream>>>(D, seg->uniq, seg->n_uniq);
  RS_CHECK_LAUNCH();
  return RS_OK;
}

RS_API int rs_shard_collect(const rs_shard *S, int64_t *recv_local, uint8_t *recv_skip, int32_t *m_total, int32_t *status,
                            void *stream) {
  ShardDev D;
  if (int rc = fill_shard(D, S, "rs_shard_collect")) return rc;
  RS_CHECK_ARG(recv_local && m_total, RS_E_ARG, "rs_shard_collect: null output");
  RS_CHECK_ARG(recv_skip || S->n_direct == 0, RS_E_ARG, "rs_shard_collect: recv_skip is required with direct ranges");
  int64_t blocks = (S->cap_recv + 255) / 256;
  const int cap = rs::num_sms() * 8;
  shard_collect_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, (cudaStream_t)stream>>>(D, recv_local, recv_skip, m_total, status);
  RS_CHECK_LAUNCH();
  return RS_OK;
}

RS_API int rs_shard_serve(const rs_shard *S, const float *table, int64_t rows, int32_t width, const int64_t *recv_local,
                          const uint8_t *skip, float *const *block, int64_t cap_block_rows, int32_t *status, void *stream) {
  ShardDev D;
  if (int rc = fill_shard(D, S, "rs_shard_serve")) return rc;
  RS_CHECK_ARG(table && rows > 0 && width >= 4 && width % 4 == 0 && recv_local && block && cap_block_rows > 0, RS_E_ARG,
               "rs_shard_serve: bad argument");
  Blocks B;
  for (int k = 0; k < S->world; ++k) {
    RS_CHECK_ARG(block[k], RS_E_ARG, "rs_shard_serve: null block pointer for rank %d", k);
    B.base[k] = block[k];
  }
  cudaStream_t st = (cudaStream_t)stream;
  const char *mode = getenv("RS_SERVE");                       // "st" forces the 128-bit load/store kernel
  const size_t smem = (size_t)SERVE_WARPS * SERVE_NST * SERVE_C * width * 4;
  if (width * 4 >= 512 && smem <= 220 * 1024 && !(mode && !strcmp(mode, "st"))) {
    RS_CUDA(cudaFuncSetAttribute(shard_serve_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    shard_serve_tma_kernel<<<rs::num_sms(), SERVE_WARPS * 32, smem, st>>>(D, table, rows, width, recv_local, skip, B, cap_block_rows, status);
  } else {
    const int wv = width / 4;
    int64_t blocks = (S->cap_recv * wv + 1023) / 1024;
    const int cap = rs::num_sms() * 8;
    shard_serve_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, st>>>(D, table, rows, wv, recv_local, skip, B, cap_block_rows, status);
  }
  RS_CHECK_LAUNCH();
  return RS_OK;
}
