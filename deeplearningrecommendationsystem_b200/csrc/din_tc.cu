// DIN / DIEN attention unit on the tensor cores (forward): score[b, l] = MLP([h, h-t, t]) for every history slot
// (reference model/din.py:39-45, model/dien.py:27-35), the two hidden layers as fused tcgen05 GEMMs.
//
// One persistent CTA per SM walks tiles of 128 (b, l) rows; thread r owns row r of the tile end to end (operand
// repack, TMEM lane, epilogues).
//   layer 0   relu((Wa + Wb) h + tb[b])        tb[b] = b0 + (Wc - Wb) t_b is precomputed per sample (din_tbias_kernel),
//             so the concat [h, h-t, t] is never built and K is D, not 3D.   MMA: M=128, N=H1, K=D  -> TMEM cols [0, H1)
//   layer 1   relu(W1 a + b1)                  the layer-0 epilogue writes relu(.) split into tf32 hi/lo STRAIGHT into
//             the A-operand chunk of the next GEMM (32 columns of D0 = one K chunk), and that chunk's MMAs are issued
//             while the next 32 columns are being read back.               MMA: M=128, N=H2, K=H1 -> TMEM cols [H1, H1+H2)
//   layer 2   w2 . relu(.) + b2                a per-row dot product in the final epilogue.
// All weights stay resident in shared memory as tf32 hi/lo pairs (3xTF32: lo*hi + hi*lo + hi*hi, ~1e-6 relative) in
// the canonical K-major core-matrix layout.  The softmax over L and the weighted sum run in din_softmax_pool_kernel;
// with pool == RS_DIN_WEIGHTS the softmax weights are the output and nothing is scaled or pooled.
#include "common.cuh"
#include "tc.cuh"

namespace {

using namespace rs::tc;
constexpr int NTH = 256;   // two warpgroups per CTA, each owning its own tiles, operand buffer, barrier and TMEM half

struct DinTcParams {
  const float *rows;  // (B, L+1, D)
  const float *tb;    // (B, H1)
  const float *W0;    // (H1, 3D)
  const float *W1;    // (H2, H1)
  const float *b1;    // (H2)
  const float *W2;    // (H2)
  const float *b2;    // (1)
  float *score;       // (B, L)
  float *act0;        // (B*L, H1) relu output of layer 0, kept for the backward (or NULL)
  float *act1;        // (B*L, H2) relu output of layer 1 (or NULL)
  int64_t B;
  int L, D, H1, H2, tmem_cols;
};

// tb[b][c] = b0[c] + sum_d (W0[c][2D+d] - W0[c][D+d]) * t_b[d]
__global__ void __launch_bounds__(128) din_tbias_kernel(const float *__restrict__ rows, const float *__restrict__ W0,
                                                        const float *__restrict__ b0, int64_t B, int L, int D, int H1,
                                                        float *__restrict__ tb) {
  extern __shared__ __align__(16) float smf[];
  float *Wt = smf;                         // [H1][D + 1]
  float *t = Wt + (size_t)H1 * (D + 1);    // [D]
  for (int e = threadIdx.x; e < H1 * D; e += blockDim.x) {
    const int c = e / D, d = e - c * D;
    Wt[c * (D + 1) + d] = W0[(size_t)c * 3 * D + 2 * D + d] - W0[(size_t)c * 3 * D + D + d];
  }
  __syncthreads();
  for (int64_t b = blockIdx.x; b < B; b += gridDim.x) {
    for (int d = threadIdx.x; d < D; d += blockDim.x) t[d] = rows[(b * (L + 1) + L) * D + d];
    __syncthreads();
    for (int c = threadIdx.x; c < H1; c += blockDim.x) {
      float acc = b0[c];
      for (int d = 0; d < D; ++d) acc = fmaf(Wt[c * (D + 1) + d], t[d], acc);
      tb[b * H1 + c] = acc;
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(NTH, 1) din_score_tc_kernel(const __grid_constant__ DinTcParams P) {
  extern __shared__ __align__(128) uint32_t sm[];
  __shared__ uint64_t bar[2];   // one per warpgroup: that group's operand buffer has been read by its MMAs
  __shared__ uint32_t tmem_base_s;
  const int warp = threadIdx.x >> 5;
  const int grp = threadIdx.x >> 7, tid = threadIdx.x & (MT - 1);   // warpgroup, row inside its tile
  const int D = P.D, H1 = P.H1, H2 = P.H2;
  uint32_t *w0h = sm, *w0l = w0h + D * H1;                    // layer 0: N = H1 rows, K = D
  uint32_t *w1h = w0l + D * H1, *w1l = w1h + H1 * H2;         // layer 1: N = H2 rows, K = H1
  uint32_t *abuf = w1l + H1 * H2;                             // [warpgroup][hi | lo][KC * MT]
  float *b1s = reinterpret_cast<float *>(abuf + 4 * KC * MT), *w2s = b1s + H2;
  if (warp == 0) tmem_alloc(&tmem_base_s, P.tmem_cols);
  if (threadIdx.x == 0) {
    rs::mbar_init(&bar[0], 1);
    rs::mbar_init(&bar[1], 1);
    rs::mbar_fence_init();
  }
  for (int e = threadIdx.x; e < D * H1; e += NTH) {
    const int n = e / D, k = e - n * D;
    const float x = P.W0[(size_t)n * 3 * D + k] + P.W0[(size_t)n * 3 * D + D + k];   // Wa + Wb
    const uint32_t h = to_tf32(x);
    w0h[tile_off(H1, n, k)] = h;
    w0l[tile_off(H1, n, k)] = to_tf32(x - __uint_as_float(h));
  }
  for (int e = threadIdx.x; e < H1 * H2; e += NTH) {
    const int n = e / H1, k = e - n * H1;
    const float x = P.W1[(size_t)n * H1 + k];
    const uint32_t h = to_tf32(x);
    w1h[tile_off(H2, n, k)] = h;
    w1l[tile_off(H2, n, k)] = to_tf32(x - __uint_as_float(h));
  }
  for (int e = threadIdx.x; e < H2; e += NTH) {
    b1s[e] = P.b1[e];
    w2s[e] = P.W2[e];
  }
  rs::fence_proxy_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = tmem_base_s + (uint32_t)grp * (uint32_t)(P.tmem_cols / 2);
  const uint32_t idesc0 = idesc_tf32(H1), idesc1 = idesc_tf32(H2);
  const uint32_t lbo_a = MT * 16, lbo_w0 = (uint32_t)H1 * 16, lbo_w1 = (uint32_t)H2 * 16, sbo = 128;
  const float b2 = P.b2[0];
  const int nchunk0 = (D + KC - 1) / KC, nchunk1 = H1 / KC;
  uint32_t uses = 0;   // commits so far on this group's barrier (-> parity of the latest phase)
  const int64_t nrows = P.B * P.L;
  const int64_t ntiles = (nrows + MT - 1) / MT;
  const int64_t first_tile = (int64_t)blockIdx.x * 2 + grp, tile_step = (int64_t)gridDim.x * 2;   // the two warpgroups take alternate tiles
  const int nS = nchunk0 + nchunk1;   // stages of one tile that read global memory: history-row chunks, tb pieces
  // Each stage's eight 16-byte pieces are fetched one stage AHEAD into `pre` (across tile boundaries too), so the
  // load latency hides behind the previous stage's repack and MMAs.
  float4 pre[KC / 4];
  auto row_of = [&](int64_t tile, int64_t &r, int64_t &b) {
    r = tile * MT + tid;
    const bool ok = r < nrows;
    b = ok ? r / P.L : 0;
    return ok;
  };
  auto prefetch = [&](int stage, bool ok, int64_t r, int64_t b) {
    const float *src;
    int n4 = KC / 4;
    if (stage < nchunk0) {
      src = P.rows + (b * (P.L + 1) + (r - b * P.L)) * D + stage * KC;
      n4 = (D - stage * KC) < KC ? (D - stage * KC) / 4 : KC / 4;
    } else {
      src = P.tb + b * H1 + (stage - nchunk0) * KC;
    }
#pragma unroll
    for (int q = 0; q < KC / 4; ++q) pre[q] = (ok && q < n4) ? rs::ldg_nc_f4(src + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
  };
  {
    int64_t r, b;
    const bool ok = row_of(first_tile, r, b);
    if (first_tile < ntiles) prefetch(0, ok, r, b);
  }
  for (int64_t tile = first_tile; tile < ntiles; tile += tile_step) {
    int64_t r, b;
    const bool valid = row_of(tile, r, b);
    int stage = 0;
    float4 cur[KC / 4];
    auto advance = [&]() {
#pragma unroll
      for (int q = 0; q < KC / 4; ++q) cur[q] = pre[q];
      ++stage;
      if (stage < nS) {
        prefetch(stage, valid, r, b);
      } else if (tile + tile_step < ntiles) {
        int64_t r2, b2;
        const bool ok2 = row_of(tile + tile_step, r2, b2);
        prefetch(0, ok2, r2, b2);
      }
    };
    // ---- layer 0: A = history rows
    for (int c = 0; c < nchunk0; ++c) {
      uint32_t *ah = abuf + (size_t)grp * 2 * KC * MT, *al = ah + KC * MT;
      advance();
      if (uses > 0) rs::mbar_wait(&bar[grp], (uses - 1) & 1u);   // the previous chunk's MMAs have read the buffer
      const int kq = (D - c * KC) < KC ? (D - c * KC) / 4 : KC / 4;   // 16-byte K pieces in this chunk
#pragma unroll
      for (int q = 0; q < KC / 4; ++q) {
        if (q < kq) {
          uint4 h, l;
          split4(cur[q], h, l);
          *reinterpret_cast<uint4 *>(ah + (q * MT + tid) * 4) = h;
          *reinterpret_cast<uint4 *>(al + (q * MT + tid) * 4) = l;
        }
      }
      rs::fence_proxy_async();
      group_sync(grp);
      if (tid == 0) {
        fence_after_sync();
        for (int s = 0; s < kq / 2; ++s) {
          const uint32_t kb = (uint32_t)(c * (KC / 4) + s * 2);
          const uint64_t dah = smem_desc(rs::smem_u32(ah) + s * 2 * lbo_a, lbo_a, sbo);
          const uint64_t dal = smem_desc(rs::smem_u32(al) + s * 2 * lbo_a, lbo_a, sbo);
          const uint64_t dbh = smem_desc(rs::smem_u32(w0h) + kb * lbo_w0, lbo_w0, sbo);
          const uint64_t dbl = smem_desc(rs::smem_u32(w0l) + kb * lbo_w0, lbo_w0, sbo);
          mma_tf32(tmem, dal, dbh, idesc0, (c == 0 && s == 0) ? 0u : 1u);
          mma_tf32(tmem, dah, dbl, idesc0, 1u);
          mma_tf32(tmem, dah, dbh, idesc0, 1u);
        }
        commit(&bar[grp]);
      }
      __syncwarp();   // warp 0 re-converges before its next aligned tcgen05.ld
      uses++;
    }
    rs::mbar_wait(&bar[grp], (uses - 1) & 1u);   // accumulator complete: the latest commit covers every earlier MMA
    fence_after_sync();
    // ---- layer 1: 32 columns of D0 -> relu(. + tb) -> one K chunk of the next A operand
    for (int c = 0; c < nchunk1; ++c) {
      uint32_t *ah = abuf + (size_t)grp * 2 * KC * MT, *al = ah + KC * MT;
      advance();
      if (uses > 0) rs::mbar_wait(&bar[grp], (uses - 1) & 1u);   // the previous chunk's MMAs have read the buffer
      uint32_t v[32];
      tmem_ld32(tmem, warp, c * KC, v);
#pragma unroll
      for (int q = 0; q < KC / 4; ++q) {
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (valid) {
          const float4 t4 = cur[q];
          x.x = fmaxf(__uint_as_float(v[4 * q + 0]) + t4.x, 0.f);
          x.y = fmaxf(__uint_as_float(v[4 * q + 1]) + t4.y, 0.f);
          x.z = fmaxf(__uint_as_float(v[4 * q + 2]) + t4.z, 0.f);
          x.w = fmaxf(__uint_as_float(v[4 * q + 3]) + t4.w, 0.f);
        }
        if (P.act0 && valid) rs::stg_cs_f4(P.act0 + r * H1 + c * KC + q * 4, x);
        uint4 h, l;
        split4(x, h, l);
        *reinterpret_cast<uint4 *>(ah + (q * MT + tid) * 4) = h;
        *reinterpret_cast<uint4 *>(al + (q * MT + tid) * 4) = l;
      }
      rs::fence_proxy_async();
      fence_before_sync();
      group_sync(grp);
      if (tid == 0) {
        fence_after_sync();
#pragma unroll
        for (int s = 0; s < KC / 8; ++s) {
          const uint32_t kb = (uint32_t)(c * (KC / 4) + s * 2);
          const uint64_t dah = smem_desc(rs::smem_u32(ah) + s * 2 * lbo_a, lbo_a, sbo);
          const uint64_t dal = smem_desc(rs::smem_u32(al) + s * 2 * lbo_a, lbo_a, sbo);
          const uint64_t dbh = smem_desc(rs::smem_u32(w1h) + kb * lbo_w1, lbo_w1, sbo);
          const uint64_t dbl = smem_desc(rs::smem_u32(w1l) + kb * lbo_w1, lbo_w1, sbo);
          mma_tf32(tmem + (uint32_t)H1, dal, dbh, idesc1, (c == 0 && s == 0) ? 0u : 1u);
          mma_tf32(tmem + (uint32_t)H1, dah, dbl, idesc1, 1u);
          mma_tf32(tmem + (uint32_t)H1, dah, dbh, idesc1, 1u);
        }
        commit(&bar[grp]);
      }
      __syncwarp();   // warp 0 re-converges before its next aligned tcgen05.ld
      uses++;
    }
    rs::mbar_wait(&bar[grp], (uses - 1) & 1u);   // accumulator complete: the latest commit covers every earlier MMA
    fence_after_sync();
    // ---- layer 2: per-row dot product over relu(D1 + b1)
    float acc = b2;
    for (int c0 = 0; c0 < H2; c0 += 32) {
      uint32_t v[32];
      tmem_ld32(tmem, warp, H1 + c0, v);
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const float a = fmaxf(__uint_as_float(v[j]) + b1s[c0 + j], 0.f);
        v[j] = __float_as_uint(a);
        acc = fmaf(w2s[c0 + j], a, acc);
      }
      if (P.act1 && valid) {
#pragma unroll
        for (int q = 0; q < 8; ++q)
          rs::stg_cs_f4(P.act1 + r * H2 + c0 + q * 4, make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]),
                                                                    __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3])));
      }
    }
    if (valid) P.score[r] = acc;
    fence_before_sync();
    group_sync(grp);   // the group's warps have drained both accumulators before its next tile's MMAs overwrite them
    fence_after_sync();
  }
  __syncthreads();
  if (warp == 0) tmem_free(tmem_base_s, P.tmem_cols);
}

// softmax over L (no mask, no scaling: model/din.py:46) and the weighted sum; one warp per sample
__global__ void __launch_bounds__(256) din_softmax_pool_kernel(const float *__restrict__ rows, const float *__restrict__ score, int64_t B,
                                                               int L, int D, int pool, float *__restrict__ out,
                                                               float *__restrict__ attw) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t b = warp_global; b < B; b += nwarps) {
    const float *s = score + b * L;
    float mx = -INFINITY;
    for (int l = lane; l < L; l += 32) mx = fmaxf(mx, s[l]);
    mx = rs::warp_max(mx);
    float sum = 0.f;
    for (int l = lane; l < L; l += 32) sum += expf(s[l] - mx);
    sum = rs::warp_sum(sum);
    const float inv = 1.f / sum;
    float *w = attw + b * L;
    for (int l = lane; l < L; l += 32) w[l] = expf(s[l] - mx) * inv;
    if (pool == RS_DIN_WEIGHTS) continue;   // attw is the output
    __syncwarp();
    const float *h = rows + b * (int64_t)(L + 1) * D;
    if (pool) {
      for (int d = lane; d < D; d += 32) {
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;   // four independent chains keep the (coalesced) loads in flight
        int l = 0;
        for (; l + 4 <= L; l += 4) {
          a0 = fmaf(w[l + 0], h[(int64_t)(l + 0) * D + d], a0);
          a1 = fmaf(w[l + 1], h[(int64_t)(l + 1) * D + d], a1);
          a2 = fmaf(w[l + 2], h[(int64_t)(l + 2) * D + d], a2);
          a3 = fmaf(w[l + 3], h[(int64_t)(l + 3) * D + d], a3);
        }
        for (; l < L; ++l) a0 = fmaf(w[l], h[(int64_t)l * D + d], a0);
        out[b * D + d] = (a0 + a1) + (a2 + a3);
      }
    } else {
      float *o = out + b * (int64_t)L * D;
      for (int e = lane; e < L * D; e += 32) o[e] = w[e / D] * h[e];
    }
  }
}

// ---------------------------------------------------------------------------------------------------- backward
// ds[b][l] = d loss / d score: softmax backward of  out = sum_l w_l h_l  (pool),  out_l = w_l h_l  or  out = w  (weights,
// g_out (B, L) = d loss / d w).  Warp per sample.
__global__ void __launch_bounds__(256) din_dscore_kernel(const float *__restrict__ rows, const float *__restrict__ attw,
                                                         const float *__restrict__ g_out, int64_t B, int L, int D, int pool,
                                                         float *__restrict__ ds) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t b = warp_global; b < B; b += nwarps) {
    const float *h = rows + b * (int64_t)(L + 1) * D;
    const float *w = attw + b * L;
    float *o = ds + b * L;
    // lane <-> history slot: dw_l = <g, h_l> from 16-byte loads (D / 4 independent loads per slot), no shuffles
    float tsum = 0.f;
    if (pool == RS_DIN_WEIGHTS) {
      for (int l = lane; l < L; l += 32) {
        const float dw = g_out[b * L + l];
        o[l] = dw;
        tsum = fmaf(w[l], dw, tsum);
      }
    } else {
      for (int l = lane; l < L; l += 32) {
        const float *g = pool ? g_out + b * D : g_out + (b * L + l) * (int64_t)D;
        const float *hl = h + (int64_t)l * D;
        float p0 = 0.f, p1 = 0.f;
        for (int q = 0; q + 8 <= D; q += 8) {
          p0 += rs::f4_dot(rs::ldg_f4(g + q), rs::ldg_nc_f4(hl + q));
          p1 += rs::f4_dot(rs::ldg_f4(g + q + 4), rs::ldg_nc_f4(hl + q + 4));
        }
        if (D & 4) p0 += rs::f4_dot(rs::ldg_f4(g + (D & ~7)), rs::ldg_nc_f4(hl + (D & ~7)));
        const float dw = p0 + p1;
        o[l] = dw;
        tsum = fmaf(w[l], dw, tsum);
      }
    }
    tsum = rs::warp_sum(tsum);
    for (int l = lane; l < L; l += 32) o[l] = w[l] * (o[l] - tsum);   // each lane re-reads only what it wrote
  }
}

struct DinTcBwdParams {
  const float *rows, *attw, *g_out, *ds;   // (B, L+1, D), (B, L), (B, D) | (B, L, D), (B, L)
  const float *act0, *act1;                // forward stashes
  const float *W0, *W1, *W2;
  float *d_rows;                           // (B, L+1, D): history rows written here, the target row by the caller
  float *dz0;                              // (B, L+1, H1): d loss / d layer-0 pre-activation, zero row at l == L
  float *dz1;                              // (B*L, H2)
  int64_t B;
  int L, D, H1, H2, pool, tmem_cols;
};

// Data-gradient chain of the attention unit, same tiling as the forward:
//   dz1 = ds w2 [a1 > 0]          (built per row, also written out for the weight-gradient GEMM)
//   da0 = dz1 W1                   MMA: M=128, N=H1, K=H2   (W1 resident as an (N=H1, K=H2) K-major image)
//   dz0 = da0 [a0 > 0]             (epilogue -> written out, and straight into the next A operand)
//   dx  = dz0 (Wa + Wb)            MMA: M=128, N=D,  K=H1   ((Wa+Wb) resident as (N=D, K=H1))
//   d_rows[b, l] = dx + w_l g      (the direct path of the weighted sum; none when the weights are the output)
__global__ void __launch_bounds__(NTH, 1) din_bwd_tc_kernel(const __grid_constant__ DinTcBwdParams P) {
  extern __shared__ __align__(128) uint32_t sm[];
  __shared__ uint64_t bar[2];   // one per warpgroup: that group's operand buffer has been read by its MMAs
  __shared__ uint32_t tmem_base_s;
  const int warp = threadIdx.x >> 5;
  const int grp = threadIdx.x >> 7, tid = threadIdx.x & (MT - 1);   // warpgroup, row inside its tile
  const int D = P.D, H1 = P.H1, H2 = P.H2;
  uint32_t *w1h = sm, *w1l = w1h + H1 * H2;                   // N = H1 rows, K = H2
  uint32_t *w0h = w1l + H1 * H2, *w0l = w0h + D * H1;         // N = D rows,  K = H1
  uint32_t *abuf = w0l + D * H1;                              // [warpgroup][hi | lo][KC * MT]
  float *w2s = reinterpret_cast<float *>(abuf + 4 * KC * MT);
  if (warp == 0) tmem_alloc(&tmem_base_s, P.tmem_cols);
  if (threadIdx.x == 0) {
    rs::mbar_init(&bar[0], 1);
    rs::mbar_init(&bar[1], 1);
    rs::mbar_fence_init();
  }
  for (int e = threadIdx.x; e < H1 * H2; e += NTH) {
    const int k = e / H1, n = e - k * H1;                     // W1 is (H2, H1): element (k = h2, n = h1), coalesced read
    const float x = P.W1[e];
    const uint32_t h = to_tf32(x);
    w1h[tile_off(H1, n, k)] = h;
    w1l[tile_off(H1, n, k)] = to_tf32(x - __uint_as_float(h));
  }
  for (int e = threadIdx.x; e < D * H1; e += NTH) {
    const int k = e / D, n = e - k * D;                       // (Wa + Wb) is (H1, D): element (k = h1, n = d)
    const float x = P.W0[(size_t)k * 3 * D + n] + P.W0[(size_t)k * 3 * D + D + n];
    const uint32_t h = to_tf32(x);
    w0h[tile_off(D, n, k)] = h;
    w0l[tile_off(D, n, k)] = to_tf32(x - __uint_as_float(h));
  }
  for (int e = threadIdx.x; e < H2; e += NTH) w2s[e] = P.W2[e];
  rs::fence_proxy_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = tmem_base_s + (uint32_t)grp * (uint32_t)(P.tmem_cols / 2);
  const uint32_t idescA = idesc_tf32(H1), idescB = idesc_tf32(D);
  const uint32_t lbo_a = MT * 16, lbo_w1 = (uint32_t)H1 * 16, lbo_w0 = (uint32_t)D * 16, sbo = 128;
  const int nchunkA = H2 / KC, nchunkB = H1 / KC;
  uint32_t uses = 0;   // commits so far on this group's barrier (-> parity of the latest phase)
  const int64_t nrows = P.B * P.L;
  const int64_t ntiles = (nrows + MT - 1) / MT;
  const int64_t first_tile = (int64_t)blockIdx.x * 2 + grp, tile_step = (int64_t)gridDim.x * 2;   // the two warpgroups take alternate tiles
  const bool direct = P.pool != RS_DIN_WEIGHTS;
  const int nG = direct ? (D + 31) / 32 : 0, nS = nchunkA + nchunkB + nG;   // stages of one tile: act1 chunks, act0 chunks, g pieces
  // Every stage consumes eight 16-byte pieces of one row of a global array.  They are fetched one stage AHEAD into
  // `pre` (across tile boundaries too), so the load latency hides behind the previous stage's repack and MMAs.
  float4 pre[KC / 4];
  float ds_pre = 0.f;
  auto row_of = [&](int64_t tile, int64_t &r, int64_t &b, int &l, int64_t &rr) {
    r = tile * MT + tid;
    const bool ok = r < nrows;
    b = ok ? r / P.L : 0;
    l = (int)(r - b * P.L);
    rr = b * (P.L + 1) + l;
    return ok;
  };
  auto prefetch = [&](int stage, bool ok, int64_t r, int64_t b) {
    const float *src;
    int n4 = KC / 4;
    if (stage < nchunkA) {
      src = P.act1 + r * H2 + stage * KC;
    } else if (stage < nchunkA + nchunkB) {
      src = P.act0 + r * H1 + (stage - nchunkA) * KC;
    } else {
      const int c0 = (stage - nchunkA - nchunkB) * 32;
      src = (P.pool ? P.g_out + b * D : P.g_out + r * D) + c0;
      n4 = (D - c0) / 4 < 8 ? (D - c0) / 4 : 8;
    }
#pragma unroll
    for (int q = 0; q < KC / 4; ++q) pre[q] = (ok && q < n4) ? rs::ldg_nc_f4(src + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
  };
  {
    int64_t r, b, rr;
    int l;
    const bool ok = row_of(first_tile, r, b, l, rr);
    if (first_tile < ntiles) {
      prefetch(0, ok, r, b);
      ds_pre = ok ? P.ds[r] : 0.f;
    }
  }
  for (int64_t tile = first_tile; tile < ntiles; tile += tile_step) {
    int64_t r, b, rr;
    int l;
    const bool valid = row_of(tile, r, b, l, rr);
    const float dsr = ds_pre;
    int stage = 0;
    float4 cur[KC / 4];
    // move the prefetched pieces into `cur` and start the loads of the next stage (or of the next tile's first)
    auto advance = [&]() {
#pragma unroll
      for (int q = 0; q < KC / 4; ++q) cur[q] = pre[q];
      ++stage;
      if (stage < nS) {
        prefetch(stage, valid, r, b);
      } else if (tile + tile_step < ntiles) {
        int64_t r2, b2, rr2;
        int l2;
        const bool ok2 = row_of(tile + tile_step, r2, b2, l2, rr2);
        prefetch(0, ok2, r2, b2);
        ds_pre = ok2 ? P.ds[r2] : 0.f;
      }
    };
    // ---- da0 = dz1 W1
    for (int c = 0; c < nchunkA; ++c) {
      uint32_t *ah = abuf + (size_t)grp * 2 * KC * MT, *al = ah + KC * MT;
      advance();
      if (uses > 0) rs::mbar_wait(&bar[grp], (uses - 1) & 1u);   // the previous chunk's MMAs have read the buffer
#pragma unroll
      for (int q = 0; q < KC / 4; ++q) {
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (valid) {
          const int k = c * KC + q * 4;
          const float4 a1 = cur[q];
          x.x = a1.x > 0.f ? dsr * w2s[k + 0] : 0.f;
          x.y = a1.y > 0.f ? dsr * w2s[k + 1] : 0.f;
          x.z = a1.z > 0.f ? dsr * w2s[k + 2] : 0.f;
          x.w = a1.w > 0.f ? dsr * w2s[k + 3] : 0.f;
          rs::stg_cs_f4(P.dz1 + r * H2 + k, x);
        }
        uint4 h, lo;
        split4(x, h, lo);
        *reinterpret_cast<uint4 *>(ah + (q * MT + tid) * 4) = h;
        *reinterpret_cast<uint4 *>(al + (q * MT + tid) * 4) = lo;
      }
      rs::fence_proxy_async();
      group_sync(grp);
      if (tid == 0) {
        fence_after_sync();
#pragma unroll
        for (int s = 0; s < KC / 8; ++s) {
          const uint32_t kb = (uint32_t)(c * (KC / 4) + s * 2);
          const uint64_t dah = smem_desc(rs::smem_u32(ah) + s * 2 * lbo_a, lbo_a, sbo);
          const uint64_t dal = smem_desc(rs::smem_u32(al) + s * 2 * lbo_a, lbo_a, sbo);
          const uint64_t dbh = smem_desc(rs::smem_u32(w1h) + kb * lbo_w1, lbo_w1, sbo);
          const uint64_t dbl = smem_desc(rs::smem_u32(w1l) + kb * lbo_w1, lbo_w1, sbo);
          mma_tf32(tmem, dal, dbh, idescA, (c == 0 && s == 0) ? 0u : 1u);
          mma_tf32(tmem, dah, dbl, idescA, 1u);
          mma_tf32(tmem, dah, dbh, idescA, 1u);
        }
        commit(&bar[grp]);
      }
      __syncwarp();
      uses++;
    }
    rs::mbar_wait(&bar[grp], (uses - 1) & 1u);   // accumulator complete: the latest commit covers every earlier MMA
    fence_after_sync();
    // ---- dz0 = da0 [a0 > 0]  ->  dx = dz0 (Wa + Wb)
    for (int c = 0; c < nchunkB; ++c) {
      uint32_t *ah = abuf + (size_t)grp * 2 * KC * MT, *al = ah + KC * MT;
      advance();
      if (uses > 0) rs::mbar_wait(&bar[grp], (uses - 1) & 1u);   // the previous chunk's MMAs have read the buffer
      uint32_t v[32];
      tmem_ld32(tmem, warp, c * KC, v);
#pragma unroll
      for (int q = 0; q < KC / 4; ++q) {
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (valid) {
          const int k = c * KC + q * 4;
          const float4 a0 = cur[q];
          x.x = a0.x > 0.f ? __uint_as_float(v[4 * q + 0]) : 0.f;
          x.y = a0.y > 0.f ? __uint_as_float(v[4 * q + 1]) : 0.f;
          x.z = a0.z > 0.f ? __uint_as_float(v[4 * q + 2]) : 0.f;
          x.w = a0.w > 0.f ? __uint_as_float(v[4 * q + 3]) : 0.f;
          rs::stg_cs_f4(P.dz0 + rr * H1 + k, x);
          if (l == P.L - 1) rs::stg_cs_f4(P.dz0 + (rr + 1) * H1 + k, make_float4(0.f, 0.f, 0.f, 0.f));   // the target slot
        }
        uint4 h, lo;
        split4(x, h, lo);
        *reinterpret_cast<uint4 *>(ah + (q * MT + tid) * 4) = h;
        *reinterpret_cast<uint4 *>(al + (q * MT + tid) * 4) = lo;
      }
      rs::fence_proxy_async();
      fence_before_sync();
      group_sync(grp);
      if (tid == 0) {
        fence_after_sync();
#pragma unroll
        for (int s = 0; s < KC / 8; ++s) {
          const uint32_t kb = (uint32_t)(c * (KC / 4) + s * 2);
          const uint64_t dah = smem_desc(rs::smem_u32(ah) + s * 2 * lbo_a, lbo_a, sbo);
          const uint64_t dal = smem_desc(rs::smem_u32(al) + s * 2 * lbo_a, lbo_a, sbo);
          const uint64_t dbh = smem_desc(rs::smem_u32(w0h) + kb * lbo_w0, lbo_w0, sbo);
          const uint64_t dbl = smem_desc(rs::smem_u32(w0l) + kb * lbo_w0, lbo_w0, sbo);
          mma_tf32(tmem + (uint32_t)H1, dal, dbh, idescB, (c == 0 && s == 0) ? 0u : 1u);
          mma_tf32(tmem + (uint32_t)H1, dah, dbl, idescB, 1u);
          mma_tf32(tmem + (uint32_t)H1, dah, dbh, idescB, 1u);
        }
        commit(&bar[grp]);
      }
      __syncwarp();
      uses++;
    }
    rs::mbar_wait(&bar[grp], (uses - 1) & 1u);   // accumulator complete: the latest commit covers every earlier MMA
    fence_after_sync();
    // ---- d_rows[b, l] = dx + w_l g,  or dx alone in the weights mode (no g stages were fetched)
    if (direct) {
      const float wl = valid ? P.attw[r] : 0.f;
      for (int c0 = 0; c0 < D; c0 += 32) {
        advance();
        uint32_t v[32];
        tmem_ld32(tmem, warp, H1 + c0, v);
        if (valid) {
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            if (c0 + 4 * q < D) {
              const float4 g4 = cur[q];
              rs::stg_f4(P.d_rows + rr * D + c0 + 4 * q,
                         make_float4(fmaf(wl, g4.x, __uint_as_float(v[4 * q + 0])), fmaf(wl, g4.y, __uint_as_float(v[4 * q + 1])),
                                     fmaf(wl, g4.z, __uint_as_float(v[4 * q + 2])), fmaf(wl, g4.w, __uint_as_float(v[4 * q + 3]))));
            }
          }
        }
      }
    } else {
      for (int c0 = 0; c0 < D; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem, warp, H1 + c0, v);
        if (valid) {
#pragma unroll
          for (int q = 0; q < 8; ++q)
            if (c0 + 4 * q < D)
              rs::stg_f4(P.d_rows + rr * D + c0 + 4 * q, make_float4(__uint_as_float(v[4 * q + 0]), __uint_as_float(v[4 * q + 1]),
                                                                      __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3])));
        }
      }
    }
    fence_before_sync();
    group_sync(grp);
    fence_after_sync();
  }
  __syncthreads();
  if (warp == 0) tmem_free(tmem_base_s, P.tmem_cols);
}

bool tc_shape_ok(int D, int H1, int H2) {
  return (D == 16 || D == 32 || D == 64) && (H1 == 64 || H1 == 128) && (H2 == 32 || H2 == 64);
}
size_t tc_smem(int D, int H1, int H2) { return ((size_t)2 * D * H1 + (size_t)2 * H1 * H2 + (size_t)4 * KC * MT + 2 * H2) * 4; }

}  // namespace

RS_API int rs_din_fwd_tc_ws_bytes(int64_t B, int32_t L, int32_t D, int32_t H1, int32_t H2, size_t *bytes) {
  RS_CHECK_ARG(bytes, RS_E_ARG, "rs_din_fwd_tc_ws_bytes: null bytes");
  RS_CHECK_ARG(tc_shape_ok(D, H1, H2), RS_E_UNSUPPORTED, "rs_din_fwd_tc: built for D in {16,32,64}, H1 in {64,128}, H2 in {32,64}");
  *bytes = ((size_t)B * H1 + (size_t)B * L) * sizeof(float);
  return RS_OK;
}

RS_API int rs_din_fwd_tc(const float *rows, int64_t B, int32_t L, int32_t D, const rs_din_weights *w, int32_t pool, float *out,
                         float *attw, float *act0, float *act1, void *ws, size_t ws_bytes, void *stream) {
  RS_CHECK_ARG(rows && w && out && w->W0 && w->b0 && w->W1 && w->b1 && w->W2 && w->b2, RS_E_ARG, "rs_din_fwd_tc: null argument");
  RS_CHECK_ARG(L >= 1, RS_E_SHAPE, "rs_din_fwd_tc: L=%d", L);
  RS_CHECK_ARG(tc_shape_ok(D, w->H1, w->H2), RS_E_UNSUPPORTED,
               "rs_din_fwd_tc: built for D in {16,32,64}, H1 in {64,128}, H2 in {32,64} (got %d, %d, %d)", D, w->H1, w->H2);
  if (B == 0) return RS_OK;
  const size_t need = ((size_t)B * w->H1 + (size_t)B * L) * sizeof(float);
  RS_CHECK_ARG(ws && ws_bytes >= need, RS_E_WORKSPACE, "rs_din_fwd_tc: workspace of %zu bytes needed, got %zu", need, ws_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  float *tb = static_cast<float *>(ws), *score = tb + (size_t)B * w->H1;
  const int sms = rs::num_sms();
  {
    const size_t smem = ((size_t)w->H1 * (D + 1) + D) * sizeof(float);
    int64_t grid = B < 2 * sms ? B : 2 * sms;
    din_tbias_kernel<<<(unsigned)grid, 128, smem, st>>>(rows, w->W0, w->b0, B, L, D, w->H1, tb);
    RS_CHECK_LAUNCH();
  }
  DinTcParams P = {};
  P.rows = rows, P.tb = tb, P.W0 = w->W0, P.W1 = w->W1, P.b1 = w->b1, P.W2 = w->W2, P.b2 = w->b2, P.score = score;
  P.act0 = act0, P.act1 = act1;
  P.B = B, P.L = L, P.D = D, P.H1 = w->H1, P.H2 = w->H2;
  P.tmem_cols = 32;
  while (P.tmem_cols < w->H1 + w->H2) P.tmem_cols <<= 1;
  P.tmem_cols *= 2;   // one half per warpgroup
  const size_t smem = tc_smem(D, w->H1, w->H2);
  RS_CUDA(cudaFuncSetAttribute(din_score_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t ntiles = (B * L + MT - 1) / MT;
  const int64_t pairs = (ntiles + 1) / 2;   // a CTA's two warpgroups take alternate tiles
  din_score_tc_kernel<<<(unsigned)(pairs < sms ? pairs : sms), NTH, smem, st>>>(P);
  RS_CHECK_LAUNCH();
  // attw doubles as the softmax output the backward needs; without it the scores are normalised in place.  In the
  // weights mode the output is that softmax output.
  float *wout = pool == RS_DIN_WEIGHTS ? out : attw ? attw : score;
  int64_t blocks = (B + 7) / 8;
  din_softmax_pool_kernel<<<(unsigned)(blocks < 8 * sms ? blocks : 8 * sms), 256, 0, st>>>(rows, score, B, L, D, pool, out, wout);
  RS_CHECK_LAUNCH();
  if (pool == RS_DIN_WEIGHTS && attw && attw != out)
    RS_CUDA(cudaMemcpyAsync(attw, out, (size_t)B * L * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return RS_OK;
}

RS_API int rs_din_bwd_tc(const float *rows, int64_t B, int32_t L, int32_t D, const rs_din_weights *w, int32_t pool,
                         const float *g_out, const float *attw, const float *act0, const float *act1, float *d_rows, float *dz0,
                         float *dz1, float *ds, void *stream) {
  RS_CHECK_ARG(rows && w && g_out && attw && act0 && act1 && d_rows && dz0 && dz1 && ds && w->W0 && w->W1 && w->W2, RS_E_ARG,
               "rs_din_bwd_tc: null argument");
  RS_CHECK_ARG(L >= 1, RS_E_SHAPE, "rs_din_bwd_tc: L=%d", L);
  RS_CHECK_ARG(tc_shape_ok(D, w->H1, w->H2), RS_E_UNSUPPORTED,
               "rs_din_bwd_tc: built for D in {16,32,64}, H1 in {64,128}, H2 in {32,64} (got %d, %d, %d)", D, w->H1, w->H2);
  if (B == 0) return RS_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int sms = rs::num_sms();
  int64_t blocks = (B + 7) / 8;
  din_dscore_kernel<<<(unsigned)(blocks < 8 * sms ? blocks : 8 * sms), 256, 0, st>>>(rows, attw, g_out, B, L, D, pool, ds);
  RS_CHECK_LAUNCH();
  DinTcBwdParams P = {};
  P.rows = rows, P.attw = attw, P.g_out = g_out, P.ds = ds, P.act0 = act0, P.act1 = act1;
  P.W0 = w->W0, P.W1 = w->W1, P.W2 = w->W2, P.d_rows = d_rows, P.dz0 = dz0, P.dz1 = dz1;
  P.B = B, P.L = L, P.D = D, P.H1 = w->H1, P.H2 = w->H2, P.pool = pool;
  P.tmem_cols = 32;
  while (P.tmem_cols < w->H1 + (D < 32 ? 32 : D)) P.tmem_cols <<= 1;
  P.tmem_cols *= 2;   // one half per warpgroup
  const size_t smem = tc_smem(D, w->H1, w->H2);
  RS_CUDA(cudaFuncSetAttribute(din_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t ntiles = (B * L + MT - 1) / MT;
  const int64_t pairs = (ntiles + 1) / 2;
  din_bwd_tc_kernel<<<(unsigned)(pairs < sms ? pairs : sms), NTH, smem, st>>>(P);
  RS_CHECK_LAUNCH();
  return RS_OK;
}
