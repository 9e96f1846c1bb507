// DIEN auxiliary loss (Zhou et al., AAAI 2019, eq. 5, inner-product form): for every sample b and t = 0..L-2,
//   x+ = <h_t, e_{t+1}>,  x- = <h_t, e^_{t+1}>,   L_aux = 1/(B (L-1)) sum_{b,t} [softplus(-x+) + softplus(x-)]
// with h_t the interest extractor's states, e_{t+1} the next clicked item and e^_{t+1} a drawn negative.
//
// The pass is HBM bound (three D-float rows read per pair in the forward; three read and three written in the
// backward), so a pair is one group of D/4 lanes holding one float4 of each row, the dot products are xor-shuffle
// trees inside the group (every lane ends with the same bits), and nothing but the rows and two floats per pair move.
// Operands are read in place from strided views: row t of sample b is at base + b * stride + t * D.
//
// The forward stashes the two loss derivatives per pair, (sigma(x+) - 1, sigma(x-)), the first computed as
// -sigma(-x+) so that it keeps its relative precision where sigma(x+) rounds to 1.  The loss is summed per block in a
// fixed order, then the block partials by one warp (rs_sigmoid_bce's scheme): bit-reproducible, no atomics.
// The backward reads the upstream gradient g from device memory (no host sync; capturable) and with c = g / (B (L-1)):
//   dh_t = c [(sigma(x+) - 1) e_{t+1} + sigma(x-) e^_{t+1}]  (t < L-1; dh_{L-1} = 0)
//   d e_{t+1} = c (sigma(x+) - 1) h_t,   d e^_{t+1} = c sigma(x-) h_t
#include "common.cuh"

namespace {

constexpr int THREADS = 256;
constexpr int MAX_PARTS = 1024;  // forward blocks = loss partials (ws floats)

__device__ __forceinline__ float softplusf_(float x) { return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x))); }
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int D>
__global__ void __launch_bounds__(THREADS) dien_aux_fwd_kernel(const float *__restrict__ h, int64_t sh, const float *__restrict__ pos,
                                                              int64_t sp, const float *__restrict__ neg, int64_t sn, int64_t B, int L,
                                                              float2 *__restrict__ sig, float *__restrict__ partial) {
  constexpr int G = D / 4;    // lanes per pair
  constexpr int PW = 32 / G;  // pairs per warp
  __shared__ float red[THREADS / 32];
  const int lane = threadIdx.x & 31, q = lane % G;
  const int64_t per = L - 1, total = B * per;
  const int64_t warp = ((int64_t)blockIdx.x * THREADS + threadIdx.x) >> 5, nwarps = (int64_t)gridDim.x * (THREADS / 32);
  float acc = 0.f;
  for (int64_t p0 = warp * PW; p0 < total; p0 += nwarps * PW) {
    const int64_t p = p0 + lane / G;
    float dp = 0.f, dn = 0.f;
    if (p < total) {
      const int64_t b = p / per, t = p - b * per;
      const float4 hv = rs::ldg_nc_f4(h + b * sh + t * D + q * 4);
      const float4 pv = rs::ldg_nc_f4(pos + b * sp + t * D + q * 4);
      const float4 nv = rs::ldg_nc_f4(neg + b * sn + t * D + q * 4);
      dp = rs::f4_dot(hv, pv);
      dn = rs::f4_dot(hv, nv);
    }
    const float xp = group_sum<G>(dp), xn = group_sum<G>(dn);
    if (p < total && q == 0) {
      sig[p] = make_float2(-sigmoidf_(-xp), sigmoidf_(xn));
      acc += softplusf_(-xp) + softplusf_(xn);
    }
  }
  acc = rs::warp_sum(acc);
  if (lane == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < THREADS / 32; ++i) s += red[i];
    partial[blockIdx.x] = s;
  }
}

__global__ void __launch_bounds__(32) dien_aux_finish_kernel(const float *__restrict__ partial, int nparts, int64_t total,
                                                            float *__restrict__ loss) {
  float s = 0.f;
  for (int i = threadIdx.x; i < nparts; i += 32) s += partial[i];
  s = rs::warp_sum(s);
  if (threadIdx.x == 0) *loss = total > 0 ? s / (float)total : 0.f;
}

template <int D>
__global__ void __launch_bounds__(THREADS) dien_aux_bwd_kernel(const float *__restrict__ h, int64_t sh, const float *__restrict__ pos,
                                                              int64_t sp, const float *__restrict__ neg, int64_t sn, int64_t B, int L,
                                                              const float2 *__restrict__ sig, const float *__restrict__ g,
                                                              float *__restrict__ dh, float *__restrict__ d_pos,
                                                              float *__restrict__ d_neg) {
  constexpr int G = D / 4;
  const int q = threadIdx.x % G;
  const int64_t per = L - 1, rows = B * L;
  const float c = per > 0 ? __ldg(g) / (float)(B * per) : 0.f;
  const int64_t grp = ((int64_t)blockIdx.x * THREADS + threadIdx.x) / G, ngrp = (int64_t)gridDim.x * (THREADS / G);
  for (int64_t r = grp; r < rows; r += ngrp) {
    const int64_t b = r / L, t = r - b * L;
    float *o = dh + r * D + q * 4;
    if (t == per) {
      rs::stg_cs_f4(o, rs::f4_zero());
      continue;
    }
    const int64_t p = b * per + t;
    const float2 s = sig[p];
    const float a = c * s.x, an = c * s.y;
    const float4 hv = rs::ldg_nc_f4(h + b * sh + t * D + q * 4);
    const float4 pv = rs::ldg_nc_f4(pos + b * sp + t * D + q * 4);
    const float4 nv = rs::ldg_nc_f4(neg + b * sn + t * D + q * 4);
    rs::stg_cs_f4(o, rs::f4_fmas(nv, an, rs::f4_scale(pv, a)));
    rs::stg_cs_f4(d_pos + p * D + q * 4, rs::f4_scale(hv, a));
    rs::stg_cs_f4(d_neg + p * D + q * 4, rs::f4_scale(hv, an));
  }
}

int check_common(const char *name, const float *h, int64_t sh, const float *pos, int64_t sp, const float *neg, int64_t sn, int64_t B,
                 int L, int D) {
  RS_CHECK_ARG(B >= 0 && L >= 1, RS_E_ARG, "%s: B=%lld L=%d", name, (long long)B, L);
  RS_CHECK_ARG(D == 16 || D == 32 || D == 64, RS_E_UNSUPPORTED, "%s: D=%d not in {16, 32, 64} (the DIN attention unit's sizes)",
               name, D);
  if (B == 0) return RS_OK;
  RS_CHECK_ARG(h && (L == 1 || (pos && neg)), RS_E_ARG, "%s: null h/pos/neg", name);
  auto aligned = [](const float *p, int64_t stride) { return ((uintptr_t)p & 15) == 0 && stride % 4 == 0; };
  RS_CHECK_ARG(aligned(h, sh) && (L == 1 || (aligned(pos, sp) && aligned(neg, sn))), RS_E_ARG,
               "%s: h/pos/neg must be 16-byte aligned with per-sample strides that are multiples of 4 floats", name);
  RS_CHECK_ARG(sh >= (int64_t)(L - 1) * D && (L == 1 || (sp >= (int64_t)(L - 1) * D && sn >= (int64_t)(L - 1) * D)), RS_E_ARG,
               "%s: per-sample stride shorter than (L-1) rows", name);
  return RS_OK;
}

int blocks_for(int64_t items, int per_block, int64_t cap) {
  const int64_t b = (items + per_block - 1) / per_block;
  return (int)(b < 1 ? 1 : (b < cap ? b : cap));
}

}  // namespace

RS_API int rs_dien_aux_fwd(const float *h, int64_t h_stride, const float *pos, int64_t pos_stride, const float *neg, int64_t neg_stride,
                           int64_t B, int32_t L, int32_t D, float *sig, float *loss, float *ws, void *stream) {
  if (int rc = check_common("rs_dien_aux_fwd", h, h_stride, pos, pos_stride, neg, neg_stride, B, L, D)) return rc;
  if (B == 0) return RS_OK;
  RS_CHECK_ARG(loss && ws && (L == 1 || sig), RS_E_ARG, "rs_dien_aux_fwd: null sig/loss/ws");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t total = B * (int64_t)(L - 1);
  int blocks = 0;
  if (total > 0) {
    blocks = blocks_for(total, THREADS / (D / 4), MAX_PARTS);
    float2 *s2 = reinterpret_cast<float2 *>(sig);
    switch (D) {
      case 16: dien_aux_fwd_kernel<16><<<blocks, THREADS, 0, st>>>(h, h_stride, pos, pos_stride, neg, neg_stride, B, L, s2, ws); break;
      case 32: dien_aux_fwd_kernel<32><<<blocks, THREADS, 0, st>>>(h, h_stride, pos, pos_stride, neg, neg_stride, B, L, s2, ws); break;
      default: dien_aux_fwd_kernel<64><<<blocks, THREADS, 0, st>>>(h, h_stride, pos, pos_stride, neg, neg_stride, B, L, s2, ws); break;
    }
    RS_CHECK_LAUNCH();
  }
  dien_aux_finish_kernel<<<1, 32, 0, st>>>(ws, blocks, total, loss);
  RS_CHECK_LAUNCH();
  return RS_OK;
}

RS_API int rs_dien_aux_bwd(const float *h, int64_t h_stride, const float *pos, int64_t pos_stride, const float *neg, int64_t neg_stride,
                           int64_t B, int32_t L, int32_t D, const float *sig, const float *g, float *dh, float *d_pos, float *d_neg,
                           void *stream) {
  if (int rc = check_common("rs_dien_aux_bwd", h, h_stride, pos, pos_stride, neg, neg_stride, B, L, D)) return rc;
  if (B == 0) return RS_OK;
  RS_CHECK_ARG(g && dh && (L == 1 || (sig && d_pos && d_neg)), RS_E_ARG, "rs_dien_aux_bwd: null sig/g/dh/d_pos/d_neg");
  RS_CHECK_ARG(((uintptr_t)dh & 15) == 0 && ((uintptr_t)d_pos & 15) == 0 && ((uintptr_t)d_neg & 15) == 0, RS_E_ARG,
               "rs_dien_aux_bwd: outputs must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t rows = B * (int64_t)L;
  const int blocks = blocks_for(rows, THREADS / (D / 4), (int64_t)rs::num_sms() * 16);
  const float2 *s2 = reinterpret_cast<const float2 *>(sig);
  switch (D) {
    case 16: dien_aux_bwd_kernel<16><<<blocks, THREADS, 0, st>>>(h, h_stride, pos, pos_stride, neg, neg_stride, B, L, s2, g, dh, d_pos, d_neg); break;
    case 32: dien_aux_bwd_kernel<32><<<blocks, THREADS, 0, st>>>(h, h_stride, pos, pos_stride, neg, neg_stride, B, L, s2, g, dh, d_pos, d_neg); break;
    default: dien_aux_bwd_kernel<64><<<blocks, THREADS, 0, st>>>(h, h_stride, pos, pos_stride, neg, neg_stride, B, L, s2, g, dh, d_pos, d_neg); break;
  }
  RS_CHECK_LAUNCH();
  return RS_OK;
}
