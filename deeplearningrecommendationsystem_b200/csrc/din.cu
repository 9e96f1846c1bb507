// DIN target attention, forward and backward (reference model/din.py:39-47; model/dien.py:27-37 with pool == 0).
//
//   z_l = [h_l, h_l - t, t];  a1 = relu(W0 z_l + b0);  a2 = relu(W1 a1 + b1);  s_l = W2 a2 + b2
//   w = softmax_l(s)  (no mask, no scaling);  out = sum_l w_l h_l  (pool),  out_l = w_l h_l  (scale)  or  out = w  (weights)
//
// The (B, L, 3D) concat never exists: with W0 = [Wa | Wb | Wc],  W0 z_l = (Wa + Wb) h_l + (Wc - Wb) t, so the
// target part is computed once per sample and the per-position part costs D*H1 instead of 3D*H1 MACs.
// One persistent CTA per SM keeps (Wa+Wb), (Wc-Wb) and W1 in shared memory (rows padded by one float so that both the
// forward, lanes over output neurons, and the backward, lanes over input features, read them conflict free) next to
// the sample's history tile and its activations.  The backward recomputes the activations, overwrites them in
// place with their gradients, and accumulates the weight gradients in registers across all samples of the CTA;
// per-CTA partials are added by the host in CTA order (deterministic).
#include "common.cuh"

namespace {

constexpr int NT = 256;

struct DinParams {
  const float *rows;  // (B, L+1, D): L history rows then the target row
  const float *W0, *b0, *W1, *b1, *W2, *b2;
  float *out, *attw;             // forward
  const float *g_out;            // backward: (B, D) pool, (B, L, D) scale or (B, L) weights
  float *d_rows;                 // (B, L+1, D) gradient through the attention only
  float *dWab_p, *dWt_p, *dW1_p, *db0_p, *db1_p, *dW2_p, *db2_p;  // per-CTA partials
  int64_t B;
  int L, pool;                   // pool: RS_DIN_SCALE, RS_DIN_WEIGHTS, any other value pools
};

template <int D, int H1, int H2>
struct Lay {
  static constexpr int WAB = 0;                         // [H1][D+1]
  static constexpr int WCB = WAB + H1 * (D + 1);        // [H1][D+1]
  static constexpr int W1P = WCB + H1 * (D + 1);        // [H2][H1+1]
  static constexpr int VEC = W1P + H2 * (H1 + 1);       // c[H1] b1[H2] W2[H2] t[D] s1[H1] red[64]
  static constexpr int C = VEC, B1 = C + H1, W2 = B1 + H2, T = W2 + H2, S1 = T + D, RED = S1 + H1, DT = RED + 64;
  static constexpr int TILE = ((DT + D + 3) / 4) * 4;   // then per-L arrays: h[L][D], a1[L][H1], a2[L][H2], s[L], w[L], dw[L]
  static size_t bytes(int L) { return (size_t)(TILE + (size_t)L * (D + H1 + H2) + 3 * ((L + 3) / 4 * 4)) * 4; }
};

__device__ __forceinline__ float block_sum(float v, float *red) {
  v = rs::warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int i = 0; i < NT / 32; ++i) t += red[i];
  __syncthreads();
  return t;
}
__device__ __forceinline__ float block_max(float v, float *red) {
  v = rs::warp_max(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = red[0];
#pragma unroll
  for (int i = 1; i < NT / 32; ++i) t = fmaxf(t, red[i]);
  __syncthreads();
  return t;
}

template <int D, int H1, int H2>
__device__ __forceinline__ void load_weights(const DinParams &P, float *sm) {
  using Y = Lay<D, H1, H2>;
  for (int e = threadIdx.x; e < H1 * D; e += NT) {
    const int j = e / D, k = e - j * D;
    const float a = P.W0[j * 3 * D + k], b = P.W0[j * 3 * D + D + k], c = P.W0[j * 3 * D + 2 * D + k];
    sm[Y::WAB + j * (D + 1) + k] = a + b;
    sm[Y::WCB + j * (D + 1) + k] = c - b;
  }
  for (int e = threadIdx.x; e < H2 * H1; e += NT) {
    const int m = e / H1, j = e - m * H1;
    sm[Y::W1P + m * (H1 + 1) + j] = P.W1[e];
  }
  for (int e = threadIdx.x; e < H2; e += NT) {
    sm[Y::B1 + e] = P.b1[e];
    sm[Y::W2 + e] = P.W2[e];
  }
}

// forward activations of one sample into shared memory; returns nothing, leaves h, a1 (post-relu), a2 (post-relu), w
template <int D, int H1, int H2>
__device__ __forceinline__ void forward_sample(const DinParams &P, float *sm, float *h, float *a1, float *a2, float *s, float *w,
                                               int64_t b) {
  using Y = Lay<D, H1, H2>;
  const int L = P.L, tid = threadIdx.x;
  const float *src = P.rows + b * (int64_t)(L + 1) * D;
  for (int e = tid; e < L * D / 4; e += NT) reinterpret_cast<float4 *>(h)[e] = rs::ldg_nc_f4(src + e * 4);
  for (int e = tid; e < D; e += NT) sm[Y::T + e] = src[(int64_t)L * D + e];
  __syncthreads();
  // target part: c[j] = b0[j] + sum_k (Wc - Wb)[j][k] t[k]
  for (int j = tid; j < H1; j += NT) {
    float acc = P.b0[j];
#pragma unroll 8
    for (int k = 0; k < D; ++k) acc = fmaf(sm[Y::WCB + j * (D + 1) + k], sm[Y::T + k], acc);
    sm[Y::C + j] = acc;
  }
  __syncthreads();
  // layer 1: a1[l][j] = relu(c[j] + sum_k (Wa+Wb)[j][k] h[l][k]);  thread (j, l-group), 4 positions at a time
  {
    constexpr int G = NT / H1;
    const int j = tid % H1, lg = tid / H1;
    const float *wj = sm + Y::WAB + j * (D + 1);
    const float cj = sm[Y::C + j];
    for (int l0 = lg * 4; l0 < L; l0 += G * 4) {
      float acc[4] = {cj, cj, cj, cj};
#pragma unroll 4
      for (int k = 0; k < D; k += 4) {
        const float w0 = wj[k], w1 = wj[k + 1], w2 = wj[k + 2], w3 = wj[k + 3];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (l0 + u < L) {
            const float4 hv = *reinterpret_cast<const float4 *>(h + (l0 + u) * D + k);
            acc[u] = fmaf(w0, hv.x, acc[u]);
            acc[u] = fmaf(w1, hv.y, acc[u]);
            acc[u] = fmaf(w2, hv.z, acc[u]);
            acc[u] = fmaf(w3, hv.w, acc[u]);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (l0 + u < L) a1[(l0 + u) * H1 + j] = fmaxf(acc[u], 0.f);
    }
  }
  __syncthreads();
  // layer 2: a2[l][m] = relu(b1[m] + sum_j W1[m][j] a1[l][j])
  {
    constexpr int G = NT / H2;
    const int m = tid % H2, lg = tid / H2;
    const float *wm = sm + Y::W1P + m * (H1 + 1);
    const float bm = sm[Y::B1 + m];
    for (int l0 = lg * 4; l0 < L; l0 += G * 4) {
      float acc[4] = {bm, bm, bm, bm};
#pragma unroll 4
      for (int j = 0; j < H1; j += 4) {
        const float w0 = wm[j], w1 = wm[j + 1], w2 = wm[j + 2], w3 = wm[j + 3];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (l0 + u < L) {
            const float4 av = *reinterpret_cast<const float4 *>(a1 + (l0 + u) * H1 + j);
            acc[u] = fmaf(w0, av.x, acc[u]);
            acc[u] = fmaf(w1, av.y, acc[u]);
            acc[u] = fmaf(w2, av.z, acc[u]);
            acc[u] = fmaf(w3, av.w, acc[u]);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (l0 + u < L) a2[(l0 + u) * H2 + m] = fmaxf(acc[u], 0.f);
    }
  }
  __syncthreads();
  // layer 3 + softmax over the L positions
  {
    const int lane = tid & 31, warp = tid >> 5;
    const float b2 = P.b2[0];
    for (int l = warp; l < L; l += NT / 32) {
      float acc = 0.f;
      for (int m = lane; m < H2; m += 32) acc = fmaf(sm[Y::W2 + m], a2[l * H2 + m], acc);
      acc = rs::warp_sum(acc);
      if (lane == 0) s[l] = acc + b2;
    }
  }
  __syncthreads();
  float mx = -INFINITY;
  for (int l = tid; l < L; l += NT) mx = fmaxf(mx, s[l]);
  mx = block_max(mx, sm + Y::RED);
  float sum = 0.f;
  for (int l = tid; l < L; l += NT) {
    const float e = expf(s[l] - mx);
    w[l] = e;
    sum += e;
  }
  sum = block_sum(sum, sm + Y::RED);
  const float inv = 1.0f / sum;
  for (int l = tid; l < L; l += NT) w[l] *= inv;
  __syncthreads();
}

template <int D, int H1, int H2>
__global__ void __launch_bounds__(NT, 1) din_fwd_kernel(const __grid_constant__ DinParams P) {
  using Y = Lay<D, H1, H2>;
  extern __shared__ __align__(16) float sm[];
  const int L = P.L, Lp = (L + 3) / 4 * 4;
  float *h = sm + Y::TILE, *a1 = h + L * D, *a2 = a1 + L * H1, *s = a2 + L * H2, *w = s + Lp;
  load_weights<D, H1, H2>(P, sm);
  __syncthreads();
  for (int64_t b = blockIdx.x; b < P.B; b += gridDim.x) {
    forward_sample<D, H1, H2>(P, sm, h, a1, a2, s, w, b);
    const int tid = threadIdx.x;
    if (P.attw)
      for (int l = tid; l < L; l += NT) P.attw[b * L + l] = w[l];
    if (P.pool == RS_DIN_WEIGHTS) {
      for (int l = tid; l < L; l += NT) P.out[b * L + l] = w[l];
    } else if (P.pool) {
      for (int d = tid; d < D; d += NT) {
        float acc = 0.f;
        for (int l = 0; l < L; ++l) acc = fmaf(w[l], h[l * D + d], acc);
        P.out[b * D + d] = acc;
      }
    } else {
      float *o = P.out + b * (int64_t)L * D;
      for (int e = tid; e < L * D; e += NT) o[e] = h[e] * w[e / D];
    }
    __syncthreads();
  }
}

template <int D, int H1, int H2>
__global__ void __launch_bounds__(NT, 1) din_bwd_kernel(const __grid_constant__ DinParams P) {
  using Y = Lay<D, H1, H2>;
  extern __shared__ __align__(16) float sm[];
  const int L = P.L, Lp = (L + 3) / 4 * 4, tid = threadIdx.x;
  float *h = sm + Y::TILE, *a1 = h + L * D, *a2 = a1 + L * H1, *s = a2 + L * H2, *w = s + Lp, *dw = w + Lp;
  load_weights<D, H1, H2>(P, sm);
  // register accumulators of the weight gradients, summed over all samples of this CTA
  constexpr int KR = D * H1 / NT;   // dWab / dWt: thread (j = tid % H1, k in [kq*KR, kq*KR+KR))
  constexpr int JR = H1 * H2 / NT;  // dW1: thread (m = tid % H2, j in [jq*JR, jq*JR+JR))
  static_assert(KR >= 4 && KR % 4 == 0 && JR >= 4 && JR % 4 == 0, "tile sizes");
  float accWab[KR], accWt[KR], accW1[JR];
#pragma unroll
  for (int i = 0; i < KR; ++i) accWab[i] = accWt[i] = 0.f;
#pragma unroll
  for (int i = 0; i < JR; ++i) accW1[i] = 0.f;
  float acc_b0 = 0.f, acc_b1 = 0.f, acc_W2 = 0.f, acc_b2 = 0.f;
  const int j6 = tid % H1, k6 = (tid / H1) * KR;
  const int m4 = tid % H2, j4 = (tid / H2) * JR;
  __syncthreads();
  for (int64_t b = blockIdx.x; b < P.B; b += gridDim.x) {
    forward_sample<D, H1, H2>(P, sm, h, a1, a2, s, w, b);
    // B1: dw[l] = <g_l, h_l>, or g_l itself when the weights are the output
    if (P.pool == RS_DIN_WEIGHTS) {
      for (int l = tid; l < L; l += NT) dw[l] = P.g_out[b * L + l];
    } else {
      const int lane = tid & 31, warp = tid >> 5;
      for (int l = warp; l < L; l += NT / 32) {
        const float *g = P.pool ? P.g_out + b * D : P.g_out + (b * L + l) * (int64_t)D;
        float acc = 0.f;
        for (int d = lane; d < D; d += 32) acc = fmaf(g[d], h[l * D + d], acc);
        acc = rs::warp_sum(acc);
        if (lane == 0) dw[l] = acc;
      }
    }
    __syncthreads();
    // B2: ds[l] = w[l] (dw[l] - sum_q w[q] dw[q])    (kept in dw)
    float part = 0.f;
    for (int l = tid; l < L; l += NT) part = fmaf(w[l], dw[l], part);
    const float tot = block_sum(part, sm + Y::RED);
    float ds_sum = 0.f;
    for (int l = tid; l < L; l += NT) {
      const float ds = w[l] * (dw[l] - tot);
      dw[l] = ds;
      ds_sum += ds;
    }
    acc_b2 += block_sum(ds_sum, sm + Y::RED);  // every thread holds the same total; thread 0's copy is written out
    // B3: dW2[m] += sum_l ds[l] a2[l][m];  a2[l][m] <- ds[l] W2[m] [a2 > 0]
    if (tid < H2) {
      float acc = 0.f;
      const float w2 = sm[Y::W2 + tid];
      for (int l = 0; l < L; ++l) {
        const float a = a2[l * H2 + tid];
        acc = fmaf(dw[l], a, acc);
        a2[l * H2 + tid] = a > 0.f ? dw[l] * w2 : 0.f;
      }
      acc_W2 += acc;
    }
    __syncthreads();
    // B4: dW1[m][j] += sum_l da2[l][m] a1[l][j];  db1[m] += sum_l da2[l][m]
    for (int l = 0; l < L; ++l) {
      const float g = a2[l * H2 + m4];
      if (j4 == 0) acc_b1 += g;
#pragma unroll
      for (int i = 0; i < JR; i += 4) {
        const float4 av = *reinterpret_cast<const float4 *>(a1 + l * H1 + j4 + i);
        accW1[i] = fmaf(g, av.x, accW1[i]);
        accW1[i + 1] = fmaf(g, av.y, accW1[i + 1]);
        accW1[i + 2] = fmaf(g, av.z, accW1[i + 2]);
        accW1[i + 3] = fmaf(g, av.w, accW1[i + 3]);
      }
    }
    __syncthreads();
    // B5: a1[l][j] <- (sum_m da2[l][m] W1[m][j]) [a1 > 0]      thread (j, l-group), 4 positions at a time
    {
      constexpr int G = NT / H1;
      const int j = tid % H1, lg = tid / H1;
      for (int l0 = lg * 4; l0 < L; l0 += G * 4) {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        for (int m = 0; m < H2; m += 4) {
          const float w0 = sm[Y::W1P + (m + 0) * (H1 + 1) + j], w1 = sm[Y::W1P + (m + 1) * (H1 + 1) + j];
          const float w2 = sm[Y::W1P + (m + 2) * (H1 + 1) + j], w3 = sm[Y::W1P + (m + 3) * (H1 + 1) + j];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            if (l0 + u < L) {
              const float4 gv = *reinterpret_cast<const float4 *>(a2 + (l0 + u) * H2 + m);
              acc[u] = fmaf(gv.x, w0, acc[u]);
              acc[u] = fmaf(gv.y, w1, acc[u]);
              acc[u] = fmaf(gv.z, w2, acc[u]);
              acc[u] = fmaf(gv.w, w3, acc[u]);
            }
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (l0 + u < L) a1[(l0 + u) * H1 + j] = a1[(l0 + u) * H1 + j] > 0.f ? acc[u] : 0.f;
      }
    }
    __syncthreads();
    // B6: dWab[j][k] += sum_l da1[l][j] h[l][k];  s1[j] = sum_l da1[l][j]
    {
      float s1 = 0.f;
      for (int l = 0; l < L; ++l) {
        const float g = a1[l * H1 + j6];
        s1 += g;
#pragma unroll
        for (int i = 0; i < KR; i += 4) {
          const float4 hv = *reinterpret_cast<const float4 *>(h + l * D + k6 + i);
          accWab[i] = fmaf(g, hv.x, accWab[i]);
          accWab[i + 1] = fmaf(g, hv.y, accWab[i + 1]);
          accWab[i + 2] = fmaf(g, hv.z, accWab[i + 2]);
          accWab[i + 3] = fmaf(g, hv.w, accWab[i + 3]);
        }
      }
      if (k6 == 0) {
        sm[Y::S1 + j6] = s1;
        acc_b0 += s1;
      }
    }
    __syncthreads();
    // B7: dWt[j][k] += s1[j] t[k];  dt[k] = sum_j s1[j] (Wc-Wb)[j][k]
    {
      const float s1 = sm[Y::S1 + j6];
#pragma unroll
      for (int i = 0; i < KR; ++i) accWt[i] = fmaf(s1, sm[Y::T + k6 + i], accWt[i]);
      for (int k = tid; k < D; k += NT) {
        float acc = 0.f;
        for (int j = 0; j < H1; ++j) acc = fmaf(sm[Y::S1 + j], sm[Y::WCB + j * (D + 1) + k], acc);
        sm[Y::DT + k] = acc;
      }
    }
    __syncthreads();
    // B8: d h[l][k] = w[l] g_l[k] + sum_j da1[l][j] (Wa+Wb)[j][k];  d target = dt.  The weights output has no direct
    // path w[l] g_l: its gradient reaches the rows through the MLP only.
    {
      float *o = P.d_rows + b * (int64_t)(L + 1) * D;
      auto chain = [&](int l, int k, float acc) {
        const float *da = a1 + l * H1;
#pragma unroll 8
        for (int j = 0; j < H1; ++j) acc = fmaf(da[j], sm[Y::WAB + j * (D + 1) + k], acc);
        return acc;
      };
      if (P.pool == RS_DIN_WEIGHTS) {
        for (int e = tid; e < L * D; e += NT) {
          const int l = e / D, k = e - l * D;
          o[e] = chain(l, k, 0.f);
        }
      } else {
        for (int e = tid; e < L * D; e += NT) {
          const int l = e / D, k = e - l * D;
          const float g = P.pool ? P.g_out[b * D + k] : P.g_out[(b * L + l) * (int64_t)D + k];
          o[e] = chain(l, k, w[l] * g);
        }
      }
      for (int k = tid; k < D; k += NT) o[(int64_t)L * D + k] = sm[Y::DT + k];
    }
    __syncthreads();
  }
  // per-CTA partials
  const int64_t c = blockIdx.x;
#pragma unroll
  for (int i = 0; i < KR; ++i) {
    P.dWab_p[(c * H1 + j6) * D + k6 + i] = accWab[i];
    P.dWt_p[(c * H1 + j6) * D + k6 + i] = accWt[i];
  }
#pragma unroll
  for (int i = 0; i < JR; ++i) P.dW1_p[(c * H2 + m4) * H1 + j4 + i] = accW1[i];
  if (k6 == 0) P.db0_p[c * H1 + j6] = acc_b0;
  if (j4 == 0) P.db1_p[c * H2 + m4] = acc_b1;
  if (tid < H2) P.dW2_p[c * H2 + tid] = acc_W2;
  if (tid == 0) P.db2_p[c] = acc_b2;
}

int grid_size(int64_t B) {
  int64_t g = rs::num_sms();
  if (g > B) g = B;
  if (g < 1) g = 1;
  return (int)g;
}

template <int D, int H1, int H2>
int launch(const DinParams &P, bool bwd, cudaStream_t st) {
  const size_t smem = Lay<D, H1, H2>::bytes(P.L);
  RS_CHECK_ARG(smem <= 227 * 1024 - 1024, RS_E_UNSUPPORTED, "rs_din: L=%d D=%d needs %zu B of shared memory", P.L, D, smem);
  const int grid = grid_size(P.B);
  if (bwd) {
    RS_CUDA(cudaFuncSetAttribute(din_bwd_kernel<D, H1, H2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    din_bwd_kernel<D, H1, H2><<<grid, NT, smem, st>>>(P);
  } else {
    RS_CUDA(cudaFuncSetAttribute(din_fwd_kernel<D, H1, H2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    din_fwd_kernel<D, H1, H2><<<grid, NT, smem, st>>>(P);
  }
  RS_CHECK_LAUNCH();
  return RS_OK;
}

int dispatch(const DinParams &P, int D, int H1, int H2, bool bwd, cudaStream_t st) {
#define RS_DIN_CASE(d, a, b) \
  if (D == d && H1 == a && H2 == b) return launch<d, a, b>(P, bwd, st);
  RS_DIN_CASE(16, 128, 64)
  RS_DIN_CASE(32, 128, 64)
  RS_DIN_CASE(64, 128, 64)
  RS_DIN_CASE(16, 64, 32)
  RS_DIN_CASE(32, 64, 32)
  RS_DIN_CASE(64, 64, 32)
#undef RS_DIN_CASE
  rs::set_error("rs_din: (D=%d, H1=%d, H2=%d) not built; D in {16,32,64}, (H1,H2) in {(128,64),(64,32)}", D, H1, H2);
  return RS_E_UNSUPPORTED;
}

}  // namespace

RS_API int rs_din_num_parts(int64_t B, int32_t *parts) {
  RS_CHECK_ARG(parts, RS_E_ARG, "rs_din_num_parts: null");
  *parts = grid_size(B);
  return RS_OK;
}

RS_API int rs_din_fwd(const float *rows, int64_t B, int32_t L, int32_t D, const rs_din_weights *w, int32_t pool, float *out,
                      float *attw, void *stream) {
  RS_CHECK_ARG(rows && w && out && L >= 1, RS_E_ARG, "rs_din_fwd: bad argument");
  if (B == 0) return RS_OK;
  DinParams P = {};
  P.rows = rows;
  P.W0 = w->W0;
  P.b0 = w->b0;
  P.W1 = w->W1;
  P.b1 = w->b1;
  P.W2 = w->W2;
  P.b2 = w->b2;
  P.out = out;
  P.attw = attw;
  P.B = B;
  P.L = L;
  P.pool = pool;
  return dispatch(P, D, w->H1, w->H2, false, (cudaStream_t)stream);
}

RS_API int rs_din_bwd(const float *rows, int64_t B, int32_t L, int32_t D, const rs_din_weights *w, int32_t pool, const float *g_out,
                      float *d_rows, float *dWab_part, float *dWt_part, float *dW1_part, float *db0_part, float *db1_part,
                      float *dW2_part, float *db2_part, int32_t num_parts, void *stream) {
  RS_CHECK_ARG(rows && w && g_out && d_rows && dWab_part && dWt_part && dW1_part && db0_part && db1_part && dW2_part && db2_part && L >= 1,
               RS_E_ARG, "rs_din_bwd: bad argument");
  RS_CHECK_ARG(num_parts == grid_size(B), RS_E_ARG, "rs_din_bwd: num_parts %d != rs_din_num_parts() = %d", num_parts, grid_size(B));
  DinParams P = {};
  P.rows = rows;
  P.W0 = w->W0;
  P.b0 = w->b0;
  P.W1 = w->W1;
  P.b1 = w->b1;
  P.W2 = w->W2;
  P.b2 = w->b2;
  P.g_out = g_out;
  P.d_rows = d_rows;
  P.dWab_p = dWab_part;
  P.dWt_p = dWt_part;
  P.dW1_p = dW1_part;
  P.db0_p = db0_part;
  P.db1_p = db1_part;
  P.dW2_p = dW2_part;
  P.db2_p = db2_part;
  P.B = B;
  P.L = L;
  P.pool = pool;
  return dispatch(P, D, w->H1, w->H2, true, (cudaStream_t)stream);
}
