// GRU recurrence (nn.GRU(D, H, batch_first=True), one layer, h0 = 0, gate order r,z,n; reference model/dien.py:47,61).
//
// The input projection gi = x.W_ih^T + b_ih is a plain GEMM over all (b, t) and is left to the library; these
// kernels own the sequential part.  A CTA keeps BT batch rows resident for all L steps: thread j holds row j of W_hh
// in registers (forward) so the per-step mat-vec gh = h.W_hh^T needs only broadcast shared-memory reads of h; the
// gate math, the state update and the stash of (r, z, n, W_hn.h + b_hn, h_t) for BPTT run in the same launch.
// Backward walks t = L-1..0 with W_hh in shared memory and emits d gi and d gh per step; the weight gradients are
// again plain GEMMs over the stashed tensors (host side).
//
// AU = true is the attention-gated form of the DIEN paper (AUGRU): with a_t = att[b, t] the update gate becomes
// u = a_t (1 - z) and h_t = (1 - u) h_{t-1} + u n, so att == 1 is nn.GRU and att == 0 keeps h == 0.  The CTA's
// BT x L attention block is staged in shared memory once (dynamic shared memory); the stash layout is unchanged
// (u is recomputed from z and a_t).  The backward also returns d_att[b, t] = sum_i dh_i (n_i - h_{t-1,i}) (1 - z_i),
// summed per (b, t) in shared memory in a fixed order, so it is bit-reproducible.
#include "common.cuh"

namespace {

constexpr int BT = 16;  // batch rows per CTA

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// gi (B, L, 3H);  h_all (B, L, H);  gates (B, L, 4H) = r | z | n | hn;  att (B, L) (AU only)
template <int H, bool AU>
__global__ void __launch_bounds__(3 * H) gru_fwd_kernel(const float *__restrict__ gi, const float *__restrict__ w_hh,
                                                       const float *__restrict__ b_hh, int64_t B, int L, float *__restrict__ h_all,
                                                       float *__restrict__ gates, const float *__restrict__ att) {
  __shared__ __align__(16) float s_h[BT][H];
  __shared__ float s_gh[BT][3 * H];
  __shared__ __align__(16) float s_gi[2][BT][3 * H];  // input projections of step t / t+1 (cp.async double buffer)
  const int j = threadIdx.x;  // gate column 0..3H-1
  float *s_att = nullptr;     // AU: [BT][L]
  if constexpr (AU) {
    extern __shared__ float s_dyn[];
    s_att = s_dyn;
  }
  float w[H];
#pragma unroll
  for (int k = 0; k < H; ++k) w[k] = w_hh[(int64_t)j * H + k];
  const float bj = b_hh[j];
  const int64_t b0 = (int64_t)blockIdx.x * BT;
  const int nb = (int)((B - b0) < BT ? (B - b0) : BT);
  for (int e = j; e < BT * H; e += 3 * H) (&s_h[0][0])[e] = 0.f;
  if constexpr (AU)
    for (int e = j; e < nb * L; e += 3 * H) s_att[e] = att[b0 * L + e];
  // the global reads of gi sit on the critical path of every step: fetch step t+1 while step t's mat-vec runs
  auto prefetch = [&](int t, int buf) {
    for (int e = j; e < nb * (3 * H / 4); e += 3 * H) {
      const int b = e / (3 * H / 4), q = e - b * (3 * H / 4);
      rs::cp_async16(&s_gi[buf][b][q * 4], gi + ((b0 + b) * L + t) * 3 * H + q * 4);
    }
    rs::cp_async_commit();
  };
  prefetch(0, 0);
  __syncthreads();
  for (int t = 0; t < L; ++t) {
    if (t + 1 < L) prefetch(t + 1, (t + 1) & 1);
    float acc[BT];
#pragma unroll
    for (int b = 0; b < BT; ++b) acc[b] = bj;
#pragma unroll
    for (int k = 0; k < H; k += 4) {
#pragma unroll
      for (int b = 0; b < BT; ++b) {
        const float4 hv = *reinterpret_cast<const float4 *>(&s_h[b][k]);  // same address for every lane: broadcast
        acc[b] = fmaf(w[k], hv.x, acc[b]);
        acc[b] = fmaf(w[k + 1], hv.y, acc[b]);
        acc[b] = fmaf(w[k + 2], hv.z, acc[b]);
        acc[b] = fmaf(w[k + 3], hv.w, acc[b]);
      }
    }
#pragma unroll
    for (int b = 0; b < BT; ++b) s_gh[b][j] = acc[b];
    if (t + 1 < L)
      rs::cp_async_wait<1>();  // step t's projections have landed (step t+1's may still be in flight)
    else
      rs::cp_async_wait<0>();
    __syncthreads();
    for (int e = j; e < nb * H; e += 3 * H) {
      const int b = e / H, i = e - b * H;
      const int64_t row = (b0 + b) * L + t;
      const float *g = &s_gi[t & 1][b][0];
      const float hr = s_gh[b][i], hz = s_gh[b][H + i], hn = s_gh[b][2 * H + i];
      const float r = sigmoidf_(g[i] + hr);
      const float z = sigmoidf_(g[H + i] + hz);
      const float n = tanhf(g[2 * H + i] + r * hn);
      const float hp = s_h[b][i];
      float hnew;
      if constexpr (AU) {
        const float u = s_att[b * L + t] * (1.0f - z);
        hnew = (1.0f - u) * hp + u * n;
      } else {
        hnew = (1.0f - z) * n + z * hp;
      }
      h_all[row * H + i] = hnew;
      if (gates) {
        float *gs = gates + row * 4 * H;
        gs[i] = r;
        gs[H + i] = z;
        gs[2 * H + i] = n;
        gs[3 * H + i] = hn;
      }
      s_h[b][i] = hnew;  // each (b,i) is touched by exactly one thread; s_gh reads above are of the old step
    }
    __syncthreads();
  }
}

// g_h_all (B, L, H) or NULL; g_h_last (B, H) or NULL.  Outputs d_gi, d_gh (B, L, 3H); AU: att (B, L) in, d_att (B, L) out.
template <int H, bool AU>
__global__ void __launch_bounds__(3 * H) gru_bwd_kernel(const float *__restrict__ w_hh, const float *__restrict__ h_all,
                                                       const float *__restrict__ gates, const float *__restrict__ g_h_all,
                                                       const float *__restrict__ g_h_last, int64_t B, int L, float *__restrict__ d_gi,
                                                       float *__restrict__ d_gh, const float *__restrict__ att,
                                                       float *__restrict__ d_att) {
  extern __shared__ float s_w[];                  // W_hh (3H, H) row-major: thread i reads column i, conflict free
  float *s_att = s_w + 3 * H * H;                 // AU: [BT][L], then the per-(b, i) terms of d_att [BT][H]
  float *s_da = s_att + BT * L;
  __shared__ float s_dh[BT][H];
  __shared__ __align__(16) float s_dgh[BT][3 * H];
  __shared__ float s_part[3][BT][H];
  const int tid = threadIdx.x;
  for (int e = tid; e < 3 * H * H; e += 3 * H) s_w[e] = w_hh[e];
  const int64_t b0 = (int64_t)blockIdx.x * BT;
  const int nb = (int)((B - b0) < BT ? (B - b0) : BT);
  for (int e = tid; e < BT * H; e += 3 * H) {
    const int b = e / H, i = e - b * H;
    (&s_dh[0][0])[e] = (g_h_last && b < nb) ? g_h_last[(b0 + b) * H + i] : 0.f;
  }
  for (int e = tid; e < BT * 3 * H; e += 3 * H) (&s_dgh[0][0])[e] = 0.f;
  if constexpr (AU)
    for (int e = tid; e < nb * L; e += 3 * H) s_att[e] = att[b0 * L + e];
  __syncthreads();
  const int part = tid / H, i = tid - part * H;   // thread (part, i): column i, gate rows [part*H, (part+1)*H)
  for (int t = L - 1; t >= 0; --t) {
    for (int e = tid; e < nb * H; e += 3 * H) {
      const int b = e / H, c = e - b * H;
      const int64_t row = (b0 + b) * L + t;
      const float *gs = gates + row * 4 * H;
      const float r = gs[c], z = gs[H + c], n = gs[2 * H + c], hn = gs[3 * H + c];
      const float hp = t > 0 ? h_all[(row - 1) * H + c] : 0.f;
      float dh = s_dh[b][c];
      if (g_h_all) dh += g_h_all[row * H + c];
      float dn, dz;
      if constexpr (AU) {
        const float a = s_att[b * L + t], u = a * (1.0f - z);
        const float du = dh * (n - hp);
        dn = dh * u;
        dz = -a * du;
        s_da[b * H + c] = du * (1.0f - z);
      } else {
        dn = dh * (1.0f - z);
        dz = dh * (hp - n);
      }
      const float dn_pre = dn * (1.0f - n * n);
      const float dz_pre = dz * z * (1.0f - z);
      const float dr_pre = dn_pre * hn * r * (1.0f - r);
      float *o1 = d_gi + row * 3 * H, *o2 = d_gh + row * 3 * H;
      o1[c] = dr_pre;
      o1[H + c] = dz_pre;
      o1[2 * H + c] = dn_pre;
      const float dghn = dn_pre * r;
      o2[c] = dr_pre;
      o2[H + c] = dz_pre;
      o2[2 * H + c] = dghn;
      s_dgh[b][c] = dr_pre;
      s_dgh[b][H + c] = dz_pre;
      s_dgh[b][2 * H + c] = dghn;
      // the direct path h_{t-1} -> h_t
      if constexpr (AU)
        s_dh[b][c] = dh * (1.0f - s_att[b * L + t] * (1.0f - z));
      else
        s_dh[b][c] = dh * z;
    }
    __syncthreads();
    // dh_prev[b][i] += sum_j dgh[b][j] * W_hh[j][i], the j range split three ways
    float acc[BT];
#pragma unroll
    for (int b = 0; b < BT; ++b) acc[b] = 0.f;
    for (int jj = 0; jj < H; jj += 4) {
      const int j = part * H + jj;
      const float w0 = s_w[(j + 0) * H + i], w1 = s_w[(j + 1) * H + i], w2 = s_w[(j + 2) * H + i], w3 = s_w[(j + 3) * H + i];
#pragma unroll
      for (int b = 0; b < BT; ++b) {
        const float4 g = *reinterpret_cast<const float4 *>(&s_dgh[b][j]);
        acc[b] = fmaf(g.x, w0, acc[b]);
        acc[b] = fmaf(g.y, w1, acc[b]);
        acc[b] = fmaf(g.z, w2, acc[b]);
        acc[b] = fmaf(g.w, w3, acc[b]);
      }
    }
#pragma unroll
    for (int b = 0; b < BT; ++b) s_part[part][b][i] = acc[b];
    __syncthreads();
    for (int e = tid; e < nb * H; e += 3 * H) {
      const int b = e / H, c = e - b * H;
      s_dh[b][c] += (s_part[0][b][c] + s_part[1][b][c]) + s_part[2][b][c];
    }
    if constexpr (AU) {
      // d_att[b, t]: one thread per sample, four interleaved partial sums over i combined in a fixed order
      if (tid < nb) {
        const float *da = s_da + tid * H;
        float p0 = 0.f, p1 = 0.f, p2 = 0.f, p3 = 0.f;
#pragma unroll
        for (int c = 0; c < H; c += 4) {
          p0 += da[c];
          p1 += da[c + 1];
          p2 += da[c + 2];
          p3 += da[c + 3];
        }
        d_att[(b0 + tid) * L + t] = (p0 + p1) + (p2 + p3);
      }
    }
    __syncthreads();
  }
}

// shared memory of the AUGRU launches: the static arrays of each kernel plus its dynamic part
constexpr size_t SMEM_MAX = 227 * 1024;
size_t fwd_smem(int L, bool au) { return au ? (size_t)BT * L * 4 : 0; }
template <int H>
size_t bwd_smem(int L, bool au) { return (size_t)3 * H * H * 4 + (au ? (size_t)BT * (L + H) * 4 : 0); }
template <int H>
bool au_smem_ok(int L) {
  return (size_t)10 * BT * H * 4 + fwd_smem(L, true) <= SMEM_MAX && (size_t)7 * BT * H * 4 + bwd_smem<H>(L, true) <= SMEM_MAX;
}

template <int H, bool AU>
int launch_fwd(const float *gi, const float *w_hh, const float *b_hh, int64_t B, int L, float *h_all, float *gates, const float *att,
               cudaStream_t st) {
  const int blocks = (int)((B + BT - 1) / BT);
  const size_t smem = fwd_smem(L, AU);
  if (AU) RS_CUDA(cudaFuncSetAttribute(gru_fwd_kernel<H, AU>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  gru_fwd_kernel<H, AU><<<blocks, 3 * H, smem, st>>>(gi, w_hh, b_hh, B, L, h_all, gates, att);
  RS_CHECK_LAUNCH();
  return RS_OK;
}
template <int H, bool AU>
int launch_bwd(const float *w_hh, const float *h_all, const float *gates, const float *g_h_all, const float *g_h_last, int64_t B, int L,
               float *d_gi, float *d_gh, const float *att, float *d_att, cudaStream_t st) {
  const int blocks = (int)((B + BT - 1) / BT);
  const size_t smem = bwd_smem<H>(L, AU);
  RS_CUDA(cudaFuncSetAttribute(gru_bwd_kernel<H, AU>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  gru_bwd_kernel<H, AU><<<blocks, 3 * H, smem, st>>>(w_hh, h_all, gates, g_h_all, g_h_last, B, L, d_gi, d_gh, att, d_att);
  RS_CHECK_LAUNCH();
  return RS_OK;
}

template <bool AU>
int dispatch_fwd(const char *name, const float *gi, const float *att, int64_t B, int L, int H, const float *w_hh, const float *b_hh,
                 float *h_all, float *gates, cudaStream_t st) {
  switch (H) {
    case 8: return launch_fwd<8, AU>(gi, w_hh, b_hh, B, L, h_all, gates, att, st);
    case 16: return launch_fwd<16, AU>(gi, w_hh, b_hh, B, L, h_all, gates, att, st);
    case 32: return launch_fwd<32, AU>(gi, w_hh, b_hh, B, L, h_all, gates, att, st);
    case 64: return launch_fwd<64, AU>(gi, w_hh, b_hh, B, L, h_all, gates, att, st);
  }
  rs::set_error("%s: hidden size %d not in {8,16,32,64}", name, H);
  return RS_E_UNSUPPORTED;
}
template <bool AU>
int dispatch_bwd(const char *name, const float *w_hh, const float *att, const float *h_all, const float *gates, const float *g_h_all,
                 const float *g_h_last, int64_t B, int L, int H, float *d_gi, float *d_gh, float *d_att, cudaStream_t st) {
  switch (H) {
    case 8: return launch_bwd<8, AU>(w_hh, h_all, gates, g_h_all, g_h_last, B, L, d_gi, d_gh, att, d_att, st);
    case 16: return launch_bwd<16, AU>(w_hh, h_all, gates, g_h_all, g_h_last, B, L, d_gi, d_gh, att, d_att, st);
    case 32: return launch_bwd<32, AU>(w_hh, h_all, gates, g_h_all, g_h_last, B, L, d_gi, d_gh, att, d_att, st);
    case 64: return launch_bwd<64, AU>(w_hh, h_all, gates, g_h_all, g_h_last, B, L, d_gi, d_gh, att, d_att, st);
  }
  rs::set_error("%s: hidden size %d not in {8,16,32,64}", name, H);
  return RS_E_UNSUPPORTED;
}

bool au_shape_ok(int L, int H) {
  switch (H) {
    case 8: return au_smem_ok<8>(L);
    case 16: return au_smem_ok<16>(L);
    case 32: return au_smem_ok<32>(L);
    case 64: return au_smem_ok<64>(L);
  }
  return true;   // the dispatch reports the hidden size
}

}  // namespace

RS_API int rs_gru_fwd(const float *gi, int64_t B, int32_t L, int32_t H, const float *w_hh, const float *b_hh, float *h_all, float *gates,
                      void *stream) {
  RS_CHECK_ARG(gi && w_hh && b_hh && h_all && B >= 0 && L >= 1, RS_E_ARG, "rs_gru_fwd: bad argument");
  if (B == 0) return RS_OK;
  return dispatch_fwd<false>("rs_gru_fwd", gi, nullptr, B, L, H, w_hh, b_hh, h_all, gates, (cudaStream_t)stream);
}

RS_API int rs_gru_bwd(const float *w_hh, const float *h_all, const float *gates, const float *g_h_all, const float *g_h_last, int64_t B,
                      int32_t L, int32_t H, float *d_gi, float *d_gh, void *stream) {
  RS_CHECK_ARG(w_hh && h_all && gates && d_gi && d_gh && (g_h_all || g_h_last) && L >= 1, RS_E_ARG, "rs_gru_bwd: bad argument");
  if (B == 0) return RS_OK;
  return dispatch_bwd<false>("rs_gru_bwd", w_hh, nullptr, h_all, gates, g_h_all, g_h_last, B, L, H, d_gi, d_gh, nullptr,
                             (cudaStream_t)stream);
}

RS_API int rs_augru_fwd(const float *gi, const float *att, int64_t B, int32_t L, int32_t H, const float *w_hh, const float *b_hh,
                        float *h_all, float *gates, void *stream) {
  RS_CHECK_ARG(gi && att && w_hh && b_hh && h_all && B >= 0 && L >= 1, RS_E_ARG, "rs_augru_fwd: bad argument");
  RS_CHECK_ARG(au_shape_ok(L, H), RS_E_UNSUPPORTED, "rs_augru_fwd: L=%d does not fit the shared-memory attention block (H=%d)", L, H);
  if (B == 0) return RS_OK;
  return dispatch_fwd<true>("rs_augru_fwd", gi, att, B, L, H, w_hh, b_hh, h_all, gates, (cudaStream_t)stream);
}

RS_API int rs_augru_bwd(const float *w_hh, const float *att, const float *h_all, const float *gates, const float *g_h_all,
                        const float *g_h_last, int64_t B, int32_t L, int32_t H, float *d_gi, float *d_gh, float *d_att, void *stream) {
  RS_CHECK_ARG(w_hh && att && h_all && gates && d_gi && d_gh && d_att && (g_h_all || g_h_last) && L >= 1, RS_E_ARG,
               "rs_augru_bwd: bad argument");
  RS_CHECK_ARG(au_shape_ok(L, H), RS_E_UNSUPPORTED, "rs_augru_bwd: L=%d does not fit the shared-memory attention block (H=%d)", L, H);
  if (B == 0) return RS_OK;
  return dispatch_bwd<true>("rs_augru_bwd", w_hh, att, h_all, gates, g_h_all, g_h_last, B, L, H, d_gi, d_gh, d_att,
                            (cudaStream_t)stream);
}
