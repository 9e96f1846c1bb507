// Shared between segment.cu (generic lane-group kernels) and segment_stream.cu (TMA-fed streaming kernel).
#pragma once
#include "common.cuh"

namespace rs {

struct UpdParams {
  const int32_t *sorted_pos, *seg_start, *seg_first_chunk, *chunk_start, *chunk_seg, *n_uniq, *n_chunks, *multi_seg, *n_multi;
  const int64_t *uniq;
  const int4 *lookup_desc;
  int32_t *work_counter;
  const int32_t *unit_start;
  float *scale_sorted;
  float *partial;
  const float *stash, *scale, *dense;
  float *table, *m, *v, *dense_grad;
  int W, F, scale_width, use_stream;
  int half_sm;       // streaming kernel: one CTA with a half-size ring per SM (leave room for a concurrent kernel)
  int combine_only;  // the chunk pass already ran elsewhere (ffm_train.cu): only add the partials of the multi-chunk segments
  Routes routes;  // routes.n > 0: RS_UPD_GRAD writes row r to a peer instead of dense_grad[r]
  float lr, wd, beta1, beta2, eps, step_size, inv_sqrt_bc2;
};

__device__ __forceinline__ float upd_sgd(float w, float g, const UpdParams &P) { return w - P.lr * (g + P.wd * w); }
__device__ __forceinline__ float4 upd_sgd(float4 w, float4 g, const UpdParams &P) {
  return make_float4(upd_sgd(w.x, g.x, P), upd_sgd(w.y, g.y, P), upd_sgd(w.z, g.z, P), upd_sgd(w.w, g.w, P));
}
// torch.optim.Adam single-tensor arithmetic on one element.  Every rounding is spelled out (the FMA contraction nvcc
// chose for the row-update kernels): left to the compiler, the same source contracts differently in different kernels
// (v = fma(g, (1-b2) g, b2 v) instead of fma(b2, v, ((1-b2) g) g)), and every kernel that calls this must give the same bits.
__device__ __forceinline__ void adam1(float &w, float &m, float &v, float g, const UpdParams &P) {
  g = __fmaf_rn(P.wd, w, g);                                          // g + wd*w
  m = __fmaf_rn(1.0f - P.beta1, __fsub_rn(g, m), m);                  // lerp_(g, 1-beta1)
  v = __fmaf_rn(P.beta2, v, __fmul_rn(__fmul_rn(1.0f - P.beta2, g), g));
  const float denom = __fmaf_rn(sqrtf(v), P.inv_sqrt_bc2, P.eps);     // sqrt(v) / sqrt(bc2) + eps
  w = __fmaf_rn(-__fdiv_rn(m, denom), P.step_size, w);                // w - step_size * m / denom
}

// Slot of a chunk's partial sum.  Full chunks are disjoint runs of RS_CHUNK sorted lookups, so start/RS_CHUNK is
// unique among them; a tail chunk (len < RS_CHUNK) is preceded by at least one full chunk of its own segment, so
// start/RS_CHUNK is unique among tails as well.  Even slots hold full chunks, odd slots tails.
__device__ __forceinline__ int partial_slot(int start, int len) { return 2 * (start / RS_CHUNK) + (len < RS_CHUNK ? 1 : 0); }

// Adam's bias-correction scalars of step u->step (and lr, wd, betas, eps) into P: the one host computation behind every
// lazy row update (rs_segment_update, rs_replica_update), so their arithmetic cannot drift apart.
void set_opt_scalars(const rs_update *u, UpdParams &P);
int fill_routes(Routes &R, const rs_routes *r, const char *who);
int launch_seg_stream(const UpdParams &P, int64_t n, int mode, cudaStream_t st);
int make_upd_params(const rs_segments *seg, int64_t n, const rs_update *u, UpdParams &P);   // segment.cu
int dispatch_update(const UpdParams &P, int mode, int64_t n, cudaStream_t st);

}  // namespace rs
