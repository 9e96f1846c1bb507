// The PNN paper's outer-product layer (OPNN with sum pooling) on the 5th-generation tensor cores.  For sample b with
// field rows e_{b,f} (D floats):  s_b = sum_f e_{b,f},  lp_b[h] = sum_{i,j} W[h, i D + j] s_b[i] s_b[j] + bias[h].
// The reference's "out" mode collapses the batch into one S^T S (gemm_tc.cu); this is the per-sample form.
//
// Every product is 3xTF32 (hi/lo operand split, three MMAs accumulated in fp32 in tensor memory), as in gemm_tc.cu.
//
// qf_kernel -- the quadratic form, used for the forward and for d lp / d S.  Both contract one operand with s_b twice,
// so both are  Acc = S_tile (128 x D) . Bop^T  (K = D) followed by a per-row contraction of Acc in the epilogue:
//   forward   Bop[n = h D + j][k = i] = W[h, i D + j]                 lp[b, h] = sum_j Acc[b, h D + j] s_b[j] + bias[h]
//   backward  Bop[n = h D + i][k = j] = W[h, i D + j] + W[h, j D + i]  dS[b, i] = sum_h g[b, h] Acc[b, h D + i]
// (the backward could also be run as g (K = H0) times Wsym (N = D^2) contracted with s_b; taking the two reductions in
// the other order costs the same MACs but keeps K = D, so the A tile stays resident and one kernel serves both).  A persistent CTA owns 128-sample tiles; thread r
// forms row r of the A tile itself (the forward sums the F field rows of E while it splits hi/lo and writes S) and owns
// TMEM lane r in the epilogue, so neither Acc nor p = s s^T reaches global memory.  Bop (H0 D rows, prepared once per
// call by prep_kernel: hi/lo, canonical K-major core-matrix order, cut into chunks of NC rows) streams from L2 through
// two shared-memory buffers filled by bulk copies; chunk q's MMAs go to TMEM accumulator q & 1, so the epilogue of chunk
// q-1 overlaps the MMAs of chunk q and the copy of chunk q+1.
//
// wgrad_kernel -- dW[h, i D + j] = sum_b g[b, h] s_b[i] s_b[j]:  A = g^T (m = h, k = b), B (n = i D + j, k = b) =
// s_b[i] s_b[j] built in shared memory from a staged 32-sample slice of S, so P (B x D^2) is never materialised.  K = B
// is cut into slabs, one CTA per (slab, 128 h, 128 n); every 512 samples the CTA adds its accumulator to its slab partial
// and restarts it.  The CTAs of the first n tile also sum g over their slab (db).
// slab_reduce_kernel adds the slab partials in slab order.  No atomics: every result is bit-identical from run to run.
#include "common.cuh"
#include "tc.cuh"

namespace {

using namespace rs::tc;
constexpr int NT = 128;   // threads per CTA: one per TMEM lane / tile row
constexpr int WN = 128;   // n columns of one wgrad CTA
constexpr int SUB = 16;   // wgrad: chunks (512 samples) per tensor-memory sum; a slab's sub-sums are added in order, so no
                          // fp32 running sum spans more than 512 samples (its rounding grows with its length)

__host__ __device__ constexpr int chunk_rows(int D) { return D == 64 ? 128 : 256; }   // NC: a chunk is <= 64 KB hi+lo

// Bop in chunks of NC rows: [chunk][hi | lo][tile_off(NC, n % NC, k)]
__global__ void prep_kernel(const float *__restrict__ W, int H0, int D, int sym, uint32_t *__restrict__ out) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // e = n D + k
  if (e >= (int64_t)H0 * D * D) return;
  const int n = (int)(e / D), k = (int)(e % D);
  const int h = n / D, c = n % D;   // c = j (forward) or i (backward)
  const float *w = W + (int64_t)h * D * D;
  const float x = sym ? w[c * D + k] + w[k * D + c] : w[k * D + c];
  const uint32_t hi = to_tf32(x), lo = to_tf32(x - __uint_as_float(hi));
  const int NC = chunk_rows(D);
  uint32_t *base = out + (int64_t)(n / NC) * 2 * NC * D;
  const int off = tile_off(NC, n % NC, k);
  base[off] = hi;
  base[NC * D + off] = lo;
}

struct QfParams {
  const float *E;        // forward: (B, F, D)
  const float *S_in;     // backward: (B, D)
  const float *G;        // backward: (B, H0)
  const uint32_t *Bop;   // prep_kernel output
  const float *bias;     // forward: (H0)
  float *out;            // forward: lp (B, H0); backward: dS (B, D)
  float *S_out;          // forward: S (B, D)
  int64_t B;
  int F, H0;
};

// chunk q of a CTA's chunk sequence (chunk q % nchunk of Bop) -> shared-memory buffer q & 1
template <int D>
__device__ __forceinline__ void load_chunk(const uint32_t *Bop, uint32_t *bbuf, uint64_t *load_bar, int64_t q, int nchunk) {
  constexpr int NC = chunk_rows(D);
  constexpr uint32_t bytes = 2u * NC * D * 4;
  uint64_t *bar = &load_bar[q & 1];
  rs::mbar_arrive_expect_tx(bar, bytes);
  rs::bulk_g2s(bbuf + (q & 1) * 2 * NC * D, Bop + (q % nchunk) * 2 * NC * D, bytes, bar);
}

template <int D, bool BWD>
__global__ void __launch_bounds__(NT, 1) qf_kernel(const __grid_constant__ QfParams P) {
  constexpr int NC = chunk_rows(D), CH = NC / D;   // Bop rows per chunk, h per chunk
  constexpr int UC = D > 32 ? D : 32, UH = UC / D;    // epilogue unit: UC accumulator columns = UH whole h
  extern __shared__ __align__(128) uint32_t sm[];
  __shared__ __align__(8) uint64_t load_bar[2], mma_bar[2];
  __shared__ uint32_t tmem_base_s;
  uint32_t *a_hi = sm, *a_lo = a_hi + MT * D, *bbuf = a_lo + MT * D;   // bbuf: [2][hi | lo][NC * D]
  const int tid = threadIdx.x, warp = tid >> 5;
  const int nchunk = P.H0 / CH;
  if (warp == 0) tmem_alloc(&tmem_base_s, 2 * NC);
  if (tid == 0) {
    for (int i = 0; i < 2; ++i) rs::mbar_init(&load_bar[i], 1), rs::mbar_init(&mma_bar[i], 1);
    rs::mbar_fence_init();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = tmem_base_s;
  const int64_t ntiles = (P.B + MT - 1) / MT;
  const int64_t total = (ntiles - 1 - blockIdx.x) / gridDim.x * nchunk + nchunk;   // chunks this CTA runs (grid <= ntiles)
  if (tid == 0)
    for (int64_t q = 0; q < 2 && q < total; ++q) load_chunk<D>(P.Bop, bbuf, load_bar, q, nchunk);
  const uint32_t idesc = idesc_tf32(NC);
  const uint32_t lbo_a = MT * 16, lbo_b = NC * 16, sbo = 128;
  int64_t q = 0;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t b = tile * MT + tid;
    const bool live = b < P.B;
    float s[D];
#pragma unroll
    for (int d = 0; d < D; ++d) s[d] = 0.f;
    if (live && !BWD) {
      const float *e = P.E + b * P.F * D;
#pragma unroll 1
      for (int f = 0; f < P.F; ++f) {
#pragma unroll
        for (int d = 0; d < D; d += 4) {
          const float4 v = rs::ldg_nc_f4(e + f * D + d);
          s[d] += v.x, s[d + 1] += v.y, s[d + 2] += v.z, s[d + 3] += v.w;
        }
      }
#pragma unroll
      for (int d = 0; d < D; d += 4) rs::stg_f4(P.S_out + b * D + d, make_float4(s[d], s[d + 1], s[d + 2], s[d + 3]));
    } else if (live) {
#pragma unroll
      for (int d = 0; d < D; d += 4) {
        const float4 v = rs::ldg_f4(P.S_in + b * D + d);
        s[d] = v.x, s[d + 1] = v.y, s[d + 2] = v.z, s[d + 3] = v.w;
      }
    }
    // A tile row tid (zero past B).  The previous tile's MMAs have all completed (its last epilogue waited for them).
#pragma unroll
    for (int d = 0; d < D; d += 4) {
      uint4 h, l;
      split4(make_float4(s[d], s[d + 1], s[d + 2], s[d + 3]), h, l);
      *reinterpret_cast<uint4 *>(a_hi + ((d >> 2) * MT + tid) * 4) = h;
      *reinterpret_cast<uint4 *>(a_lo + ((d >> 2) * MT + tid) * 4) = l;
    }
    rs::fence_proxy_async();
    __syncthreads();
    float acc[BWD ? D : 1];
#pragma unroll
    for (int d = 0; d < (BWD ? D : 1); ++d) acc[d] = 0.f;

    for (int c = 0; c <= nchunk; ++c, ++q) {   // MMAs of chunk c, then the epilogue of chunk c - 1
      if (tid == 0 && c < nchunk) {
        const int bi = (int)(q & 1);
        rs::mbar_wait(&load_bar[bi], (uint32_t)(q >> 1) & 1u);
        fence_after_sync();
        const uint32_t bh = rs::smem_u32(bbuf + bi * 2 * NC * D), bl = bh + NC * D * 4;
        const uint32_t ah = rs::smem_u32(a_hi), al = rs::smem_u32(a_lo);
#pragma unroll
        for (int k = 0; k < D / 8; ++k) {   // one MMA covers K = 8 = two 16-byte K halves
          const uint32_t oa = k * 2 * lbo_a, ob = k * 2 * lbo_b;
          const uint64_t dah = smem_desc(ah + oa, lbo_a, sbo), dal = smem_desc(al + oa, lbo_a, sbo);
          const uint64_t dbh = smem_desc(bh + ob, lbo_b, sbo), dbl = smem_desc(bl + ob, lbo_b, sbo);
          const uint32_t d_tmem = tmem + bi * NC;
          mma_tf32(d_tmem, dal, dbh, idesc, k ? 1u : 0u);   // small terms first
          mma_tf32(d_tmem, dah, dbl, idesc, 1u);
          mma_tf32(d_tmem, dah, dbh, idesc, 1u);
        }
        commit(&mma_bar[bi]);
      }
      if (c == 0) continue;
      // epilogue of chunk c - 1 (sequence index p): contract accumulator p & 1 with s_b (forward) or g_b (backward)
      const int64_t p = q - 1;
      const int bi = (int)(p & 1), h0 = (c - 1) * CH;
      rs::mbar_wait(&mma_bar[bi], (uint32_t)(p >> 1) & 1u);
      fence_after_sync();
      if (tid == 0 && p + 2 < total) load_chunk<D>(P.Bop, bbuf, load_bar, p + 2, nchunk);   // chunk p's MMAs have read its buffer
      __syncwarp();
#pragma unroll 1
      for (int u = 0; u < NC / UC; ++u) {   // UC columns = UH whole h
        float gv[UH], r[UH];
#pragma unroll
        for (int hh = 0; hh < UH; ++hh) r[hh] = 0.f, gv[hh] = (BWD && live) ? P.G[b * P.H0 + h0 + u * UH + hh] : 0.f;
#pragma unroll
        for (int c0 = 0; c0 < UC; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(tmem + bi * NC, warp, u * UC + c0, v);
#pragma unroll
          for (int jj = 0; jj < 32; ++jj) {
            const int hh = (c0 + jj) / D, j = (c0 + jj) % D;
            if (BWD)
              acc[j] = fmaf(gv[hh], __uint_as_float(v[jj]), acc[j]);
            else
              r[hh] = fmaf(__uint_as_float(v[jj]), s[j], r[hh]);
          }
        }
        if (!BWD && live) {
#pragma unroll
          for (int hh = 0; hh < UH; ++hh) P.out[b * P.H0 + h0 + u * UH + hh] = r[hh] + P.bias[h0 + u * UH + hh];
        }
      }
      fence_before_sync();
      __syncthreads();   // every lane has read accumulator bi before chunk p + 2's MMAs overwrite it
      fence_after_sync();
    }
    --q;   // the last pass issued no chunk
    if (BWD && live) {
#pragma unroll
      for (int d = 0; d < D; d += 4) rs::stg_f4(P.out + b * D + d, make_float4(acc[d], acc[d + 1], acc[d + 2], acc[d + 3]));
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_free(tmem, 2 * NC);
}

// slab z, h tile blockIdx.y, n tile blockIdx.x -> partial + z * (H0 D^2 + H0): [dW (H0, D^2) | db (H0)]
template <int D>
__global__ void __launch_bounds__(NT, 3) wgrad_kernel(const float *__restrict__ G, const float *__restrict__ S, int64_t B, int H0,
                                                      int64_t slab, float *__restrict__ partial) {
  extern __shared__ __align__(128) uint32_t sm[];
  __shared__ float s_s[KC][D];
  __shared__ uint64_t mma_bar;
  __shared__ uint32_t tmem_base_s;
  uint32_t *a_hi = sm, *a_lo = a_hi + KC * MT, *b_hi = a_lo + KC * MT, *b_lo = b_hi + KC * WN;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (warp == 0) tmem_alloc(&tmem_base_s, WN);
  if (tid == 0) {
    rs::mbar_init(&mma_bar, 1);
    rs::mbar_fence_init();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = tmem_base_s;
  const uint32_t idesc = idesc_tf32(WN);
  const uint32_t lbo_a = MT * 16, lbo_b = WN * 16, sbo = 128;
  const int h = blockIdx.y * MT + tid;
  const bool hv = h < H0;
  const int n = blockIdx.x * WN + tid, i = n / D, j = n % D;   // this thread's B row
  const int64_t k_lo = (int64_t)blockIdx.z * slab, k_hi = k_lo + slab < B ? k_lo + slab : B;
  const int64_t stride = (int64_t)H0 * D * D + H0;
  float *dst = partial + blockIdx.z * stride;
  const int row = blockIdx.y * MT + warp * 32 + lane;   // == h
  float gsum = 0.f;
  uint32_t phase = 0;
  int nc = 0;   // chunks accumulated so far
  for (int64_t k0 = k_lo; k0 < k_hi; k0 += KC, ++nc) {
    for (int e = tid; e < KC * D; e += NT) {
      const int kk = e / D;
      s_s[kk][e % D] = k0 + kk < k_hi ? S[(k0 + kk) * D + e % D] : 0.f;
    }
    float v[KC];
#pragma unroll
    for (int kk = 0; kk < KC; ++kk) v[kk] = (hv && k0 + kk < k_hi) ? G[(k0 + kk) * H0 + h] : 0.f;
    if (blockIdx.x == 0) {
#pragma unroll
      for (int kk = 0; kk < KC; ++kk) gsum += v[kk];
    }
#pragma unroll
    for (int q = 0; q < KC / 4; ++q) {
      uint4 hi, lo;
      split4(make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]), hi, lo);
      *reinterpret_cast<uint4 *>(a_hi + (q * MT + tid) * 4) = hi;
      *reinterpret_cast<uint4 *>(a_lo + (q * MT + tid) * 4) = lo;
    }
    __syncthreads();   // s_s staged
#pragma unroll
    for (int q = 0; q < KC / 4; ++q) {
      const float4 p = make_float4(s_s[4 * q][i] * s_s[4 * q][j], s_s[4 * q + 1][i] * s_s[4 * q + 1][j],
                                   s_s[4 * q + 2][i] * s_s[4 * q + 2][j], s_s[4 * q + 3][i] * s_s[4 * q + 3][j]);
      uint4 hi, lo;
      split4(p, hi, lo);
      *reinterpret_cast<uint4 *>(b_hi + (q * WN + tid) * 4) = hi;
      *reinterpret_cast<uint4 *>(b_lo + (q * WN + tid) * 4) = lo;
    }
    rs::fence_proxy_async();
    __syncthreads();
    if (tid == 0) {
      fence_after_sync();
#pragma unroll
      for (int s = 0; s < KC / 8; ++s) {
        const uint64_t ah = smem_desc(rs::smem_u32(a_hi) + s * 2 * lbo_a, lbo_a, sbo);
        const uint64_t al = smem_desc(rs::smem_u32(a_lo) + s * 2 * lbo_a, lbo_a, sbo);
        const uint64_t bh = smem_desc(rs::smem_u32(b_hi) + s * 2 * lbo_b, lbo_b, sbo);
        const uint64_t bl = smem_desc(rs::smem_u32(b_lo) + s * 2 * lbo_b, lbo_b, sbo);
        mma_tf32(tmem, al, bh, idesc, (nc % SUB == 0 && s == 0) ? 0u : 1u);
        mma_tf32(tmem, ah, bl, idesc, 1u);
        mma_tf32(tmem, ah, bh, idesc, 1u);
      }
      commit(&mma_bar);
    }
    __syncwarp();
    rs::mbar_wait(&mma_bar, phase);   // the MMAs have read shared memory: the next chunk may overwrite it
    phase ^= 1u;
    fence_after_sync();
    if ((nc + 1) % SUB == 0 || k0 + KC >= k_hi) {   // flush the sub-sum: partial row (+)= accumulator row
      const bool first = nc < SUB;
#pragma unroll 1
      for (int c0 = 0; c0 < WN; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem, warp, c0, v);
        if (row < H0) {
          float *o = dst + (int64_t)row * D * D + blockIdx.x * WN + c0;
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float4 x = make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]),
                                   __uint_as_float(v[4 * q + 3]));
            if (!first) x = rs::f4_add(rs::ldg_f4(o + 4 * q), x);
            rs::stg_f4(o + 4 * q, x);
          }
        }
      }
      fence_before_sync();   // the next chunk's first MMA overwrites the accumulator after the next __syncthreads
    }
  }
  if (blockIdx.x == 0 && hv) dst[(int64_t)H0 * D * D + h] = gsum;
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_free(tmem, WN);
}

__global__ void slab_reduce_kernel(const float *__restrict__ partial, int nslabs, int64_t nw, int H0, float *__restrict__ dW,
                                   float *__restrict__ db) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = nw + H0;
  if (e >= stride) return;
  float acc = 0.f;
  for (int z = 0; z < nslabs; ++z) acc += partial[z * stride + e];
  if (e < nw)
    dW[e] = acc;
  else
    db[e - nw] = acc;
}

// K = B in slabs of whole 32-sample chunks: about 3 CTAs per SM over the (h, n) output tiles
int plan_slabs(int64_t B, int D, int H0, int64_t *slab) {
  const int64_t tiles = (int64_t)((H0 + MT - 1) / MT) * (D * D / WN);
  const int64_t chunks = (B + KC - 1) / KC;
  int64_t n = (int64_t)rs::num_sms() * 3 / tiles;
  if (n > chunks) n = chunks;
  if (n < 1) n = 1;
  const int64_t per = (chunks + n - 1) / n;
  *slab = per * KC;
  return (int)((chunks + per - 1) / per);
}

size_t prep_bytes(int D, int H0) { return (size_t)2 * H0 * D * D * 4; }
size_t partial_offset(int D, int H0) { return (prep_bytes(D, H0) + 255) / 256 * 256; }

int check_shape(const char *who, int64_t B, int D, int H0) {
  RS_CHECK_ARG(B >= 0, RS_E_ARG, "%s: bad argument (B = %lld)", who, (long long)B);
  RS_CHECK_ARG(D == 16 || D == 32 || D == 64, RS_E_UNSUPPORTED, "%s: D must be 16, 32 or 64 (got %d)", who, D);
  RS_CHECK_ARG(H0 >= 16 && H0 <= 512 && H0 % 16 == 0, RS_E_UNSUPPORTED, "%s: H0 must be a multiple of 16 in [16, 512] (got %d)", who, H0);
  return RS_OK;
}

bool aligned16(const void *p) { return ((uintptr_t)p & 15) == 0; }

template <int D, bool BWD>
int launch_qf(const QfParams &P, cudaStream_t st) {
  constexpr int NC = chunk_rows(D);
  const size_t smem = (size_t)(2 * MT * D + 2 * 2 * NC * D) * 4;
  RS_CUDA(cudaFuncSetAttribute(qf_kernel<D, BWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t ntiles = (P.B + MT - 1) / MT;
  const int grid = (int)(ntiles < rs::num_sms() ? ntiles : rs::num_sms());
  qf_kernel<D, BWD><<<grid, NT, smem, st>>>(P);
  RS_CHECK_LAUNCH();
  return RS_OK;
}

int prep(const float *W, int D, int H0, int sym, uint32_t *out, cudaStream_t st) {
  const int64_t n = (int64_t)H0 * D * D;
  prep_kernel<<<(int)((n + 255) / 256), 256, 0, st>>>(W, H0, D, sym, out);
  RS_CHECK_LAUNCH();
  return RS_OK;
}

template <int D>
int launch_wgrad(const float *g, const float *S, int64_t B, int H0, float *partial, float *dW, float *db, cudaStream_t st) {
  int64_t slab;
  const int nslabs = plan_slabs(B, D, H0, &slab);
  const size_t smem = (size_t)(2 * KC * MT + 2 * KC * WN) * 4;
  RS_CUDA(cudaFuncSetAttribute(wgrad_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const dim3 grid(D * D / WN, (H0 + MT - 1) / MT, nslabs);
  wgrad_kernel<D><<<grid, NT, smem, st>>>(g, S, B, H0, slab, partial);
  RS_CHECK_LAUNCH();
  const int64_t stride = (int64_t)H0 * D * D + H0;
  slab_reduce_kernel<<<(int)((stride + 255) / 256), 256, 0, st>>>(partial, nslabs, (int64_t)H0 * D * D, H0, dW, db);
  RS_CHECK_LAUNCH();
  return RS_OK;
}

}  // namespace

RS_API int rs_pnn_outer_ws_bytes(int64_t B, int32_t D, int32_t H0, size_t *fwd_bytes, size_t *bwd_bytes) {
  RS_CHECK_ARG(fwd_bytes && bwd_bytes, RS_E_ARG, "rs_pnn_outer_ws_bytes: null output pointer");
  const int rc = check_shape("rs_pnn_outer_ws_bytes", B, D, H0);
  if (rc) return rc;
  int64_t slab;
  const int nslabs = B > 0 ? plan_slabs(B, D, H0, &slab) : 0;
  *fwd_bytes = prep_bytes(D, H0);
  *bwd_bytes = partial_offset(D, H0) + (size_t)nslabs * ((size_t)H0 * D * D + H0) * 4;
  return RS_OK;
}

RS_API int rs_pnn_outer_fwd(const float *E, int64_t B, int32_t F, int32_t D, int32_t H0, const float *W, const float *bias, float *lp,
                            float *S, void *ws, size_t ws_bytes, void *stream) {
  RS_CHECK_ARG(E && W && bias && lp && S && ws && F >= 1, RS_E_ARG, "rs_pnn_outer_fwd: bad argument (null pointer or F < 1)");
  const int rc = check_shape("rs_pnn_outer_fwd", B, D, H0);
  if (rc) return rc;
  RS_CHECK_ARG(aligned16(E) && aligned16(S) && aligned16(ws), RS_E_ARG, "rs_pnn_outer_fwd: E, S and ws must be 16-byte aligned");
  RS_CHECK_ARG(ws_bytes >= prep_bytes(D, H0), RS_E_WORKSPACE, "rs_pnn_outer_fwd: workspace too small");
  if (B == 0) return RS_OK;
  cudaStream_t st = (cudaStream_t)stream;
  uint32_t *bop = (uint32_t *)ws;
  int r = prep(W, D, H0, 0, bop, st);
  if (r) return r;
  QfParams P = {};
  P.E = E, P.Bop = bop, P.bias = bias, P.out = lp, P.S_out = S, P.B = B, P.F = F, P.H0 = H0;
  return D == 16 ? launch_qf<16, false>(P, st) : D == 32 ? launch_qf<32, false>(P, st) : launch_qf<64, false>(P, st);
}

RS_API int rs_pnn_outer_bwd(const float *S, const float *g, int64_t B, int32_t D, int32_t H0, const float *W, float *dS, float *dW,
                            float *db, void *ws, size_t ws_bytes, void *stream) {
  RS_CHECK_ARG(S && g && W && dS && dW && db && ws, RS_E_ARG, "rs_pnn_outer_bwd: bad argument (null pointer)");
  const int rc = check_shape("rs_pnn_outer_bwd", B, D, H0);
  if (rc) return rc;
  RS_CHECK_ARG(aligned16(S) && aligned16(dS) && aligned16(ws), RS_E_ARG, "rs_pnn_outer_bwd: S, dS and ws must be 16-byte aligned");
  size_t fwd_need, need;
  rs_pnn_outer_ws_bytes(B, D, H0, &fwd_need, &need);
  RS_CHECK_ARG(ws_bytes >= need, RS_E_WORKSPACE, "rs_pnn_outer_bwd: workspace too small (%zu < %zu bytes)", ws_bytes, need);
  cudaStream_t st = (cudaStream_t)stream;
  if (B == 0) {   // empty batch: zero gradients
    RS_CUDA(cudaMemsetAsync(dW, 0, (size_t)H0 * D * D * 4, st));
    RS_CUDA(cudaMemsetAsync(db, 0, (size_t)H0 * 4, st));
    return RS_OK;
  }
  uint32_t *bop = (uint32_t *)ws;
  float *partial = (float *)((char *)ws + partial_offset(D, H0));
  int r = prep(W, D, H0, 1, bop, st);
  if (r) return r;
  QfParams P = {};
  P.S_in = S, P.G = g, P.Bop = bop, P.out = dS, P.B = B, P.H0 = H0;
  r = D == 16 ? launch_qf<16, true>(P, st) : D == 32 ? launch_qf<32, true>(P, st) : launch_qf<64, true>(P, st);
  if (r) return r;
  return D == 16 ? launch_wgrad<16>(g, S, B, H0, partial, dW, db, st)
         : D == 32 ? launch_wgrad<32>(g, S, B, H0, partial, dW, db, st)
                   : launch_wgrad<64>(g, S, B, H0, partial, dW, db, st);
}
