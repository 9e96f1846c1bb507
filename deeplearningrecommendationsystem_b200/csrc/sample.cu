// Input preparation on the device (SURVEY.md 8(f).2): negative sampling and feature-matrix assembly.
//
// rs_sample_negatives is the device counterpart of sampler/sampler.py:16-27 (for every user, num_negatives items drawn
// uniformly, redrawn while (user, item) is an observed pair).  The reference consumes python's global `random`
// sequentially, which no parallel sampler can replay, so the host-side Sampler stays the bit-exact path and this one
// is OPTIONAL: same acceptance rule, its own documented stream -- Philox4x32-10 keyed by the seed, counter =
// (sample index, attempt block, call epoch) -- so every (user, slot) is a pure function of (seed, epoch) regardless of
// scheduling, and the numpy restatement in oracle/sampling.py reproduces it bit for bit.
//
// rs_dien_negatives draws the negatives of DIEN's auxiliary loss on the same stream (an extension: the reference has no
// auxiliary loss), one slot per (sample, history position), redrawn while equal to the clicked item.
//
// rs_assemble_features is data/reader.py:98-101 (`pd.merge` with the user and the item side-feature tables):
// row b = [user, item, user_feat[user, :], item_feat[item, :]] as fp32, one coalesced pass.
#include "common.cuh"

namespace rs {
namespace {

struct Philox {
  uint32_t c[4];
};
__device__ __forceinline__ Philox philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return Philox{{c0, c1, c2, c3}};
}

__device__ __forceinline__ bool contains(const int64_t *__restrict__ keys, int64_t n, int64_t key) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    int64_t v = keys[mid];
    if (v < key) lo = mid + 1;
    else hi = mid;
  }
  return lo < n && keys[lo] == key;
}

constexpr uint32_t MAX_BLOCKS = 1u << 14;  // 65536 attempts before a slot gives up (user with ~every item observed)

__global__ void sample_negatives_kernel(const int64_t *__restrict__ excl, int64_t n_excl, int64_t num_user, int64_t num_item,
                                        int32_t per_user, uint32_t seed_lo, uint32_t seed_hi, uint32_t epoch,
                                        int64_t *__restrict__ out_users, int64_t *__restrict__ out_items, int32_t *status) {
  const int64_t total = num_user * per_user;
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < total; s += (int64_t)gridDim.x * blockDim.x) {
    const int64_t user = s / per_user;
    int64_t item = -1;
    for (uint32_t blk = 0; blk < MAX_BLOCKS && item < 0; ++blk) {
      Philox p = philox4x32_10((uint32_t)s, (uint32_t)(s >> 32), blk, epoch, seed_lo, seed_hi);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (item < 0) {
          int64_t cand = (int64_t)(((uint64_t)p.c[j] * (uint64_t)num_item) >> 32);
          if (!contains(excl, n_excl, user * num_item + cand)) item = cand;
        }
      }
    }
    if (item < 0) {
      atomicOr(status, 8);
      item = 0;
    }
    out_users[s] = user;
    out_items[s] = item;
  }
}

// DIEN auxiliary-loss negatives: slot s = b (L-1) + t draws a uniform item for position t+1 of sample b, redrawn while it
// equals hist[b, t+1].  The epoch is read from device memory, so a graph-replayed step that advances it on the device
// draws a fresh set on every replay.
__global__ void dien_negatives_kernel(const int64_t *__restrict__ hist, int64_t B, int L, int64_t num_item, uint32_t seed_lo,
                                      uint32_t seed_hi, const int64_t *__restrict__ epoch_p, int64_t *__restrict__ neg,
                                      int32_t *status) {
  const int64_t per = L - 1, total = B * per;
  const uint32_t epoch = (uint32_t)*epoch_p;
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < total; s += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = s / per, t = s - b * per;
    const int64_t pos = clamp_id(hist[b * L + t + 1], num_item, status);
    int64_t item = -1;
    for (uint32_t blk = 0; blk < MAX_BLOCKS && item < 0; ++blk) {
      Philox p = philox4x32_10((uint32_t)s, (uint32_t)(s >> 32), blk, epoch, seed_lo, seed_hi);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t cand = (int64_t)(((uint64_t)p.c[j] * (uint64_t)num_item) >> 32);
        if (item < 0 && cand != pos) item = cand;
      }
    }
    if (item < 0) {
      atomicOr(status, 8);
      item = pos + 1 < num_item ? pos + 1 : 0;
    }
    neg[s] = item;
  }
}

__global__ void assemble_features_kernel(const int64_t *__restrict__ users, const int64_t *__restrict__ items,
                                         const float *__restrict__ user_feat, int64_t num_user, int FU,
                                         const float *__restrict__ item_feat, int64_t num_item, int FI, int64_t B,
                                         float *__restrict__ out, int32_t *status) {
  const int W = 2 + FU + FI;
  const int64_t total = B * W;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = e / W;
    const int c = (int)(e - b * W);
    float v;
    if (c == 0) {
      v = (float)users[b];
    } else if (c == 1) {
      v = (float)items[b];
    } else if (c < 2 + FU) {
      v = user_feat[clamp_id(users[b], num_user, status) * FU + (c - 2)];
    } else {
      v = item_feat[clamp_id(items[b], num_item, status) * FI + (c - 2 - FU)];
    }
    out[e] = v;
  }
}

}  // namespace
}  // namespace rs

RS_API int rs_sample_negatives(const int64_t *excluded_keys, int64_t num_excluded, int64_t num_user, int64_t num_item,
                               int32_t num_negatives, uint64_t seed, uint32_t epoch, int64_t *out_users, int64_t *out_items,
                               int32_t *status, void *stream) {
  using namespace rs;
  RS_CHECK_ARG(num_user >= 0 && num_negatives >= 0, RS_E_ARG, "rs_sample_negatives: num_user=%lld num_negatives=%d",
               (long long)num_user, num_negatives);
  RS_CHECK_ARG(num_item >= 1 && num_item < (1ll << 32), RS_E_ARG, "rs_sample_negatives: num_item=%lld outside [1, 2^32)",
               (long long)num_item);
  RS_CHECK_ARG(num_excluded == 0 || excluded_keys, RS_E_ARG, "rs_sample_negatives: null excluded_keys");
  const int64_t total = num_user * num_negatives;
  if (total == 0) return 0;
  RS_CHECK_ARG(out_users && out_items && status, RS_E_ARG, "rs_sample_negatives: null outputs/status");
  int64_t blocks = (total + 255) / 256;
  int64_t cap = (int64_t)num_sms() * 16;
  sample_negatives_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, (cudaStream_t)stream>>>(
      excluded_keys, num_excluded, num_user, num_item, num_negatives, (uint32_t)seed, (uint32_t)(seed >> 32), epoch, out_users,
      out_items, status);
  RS_CHECK_LAUNCH();
  return 0;
}

RS_API int rs_dien_negatives(const int64_t *hist, int64_t B, int32_t L, int64_t num_item, uint64_t seed, const int64_t *epoch,
                             int64_t *neg, int32_t *status, void *stream) {
  using namespace rs;
  RS_CHECK_ARG(B >= 0 && L >= 1, RS_E_ARG, "rs_dien_negatives: B=%lld L=%d", (long long)B, L);
  RS_CHECK_ARG(num_item >= 2 && num_item < (1ll << 32), RS_E_ARG, "rs_dien_negatives: num_item=%lld outside [2, 2^32)",
               (long long)num_item);
  const int64_t total = B * (L - 1);
  if (total == 0) return 0;
  RS_CHECK_ARG(hist && epoch && neg && status, RS_E_ARG, "rs_dien_negatives: null hist/epoch/neg/status");
  int64_t blocks = (total + 255) / 256;
  int64_t cap = (int64_t)num_sms() * 16;
  dien_negatives_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, (cudaStream_t)stream>>>(
      hist, B, L, num_item, (uint32_t)seed, (uint32_t)(seed >> 32), epoch, neg, status);
  RS_CHECK_LAUNCH();
  return 0;
}

RS_API int rs_assemble_features(const int64_t *users, const int64_t *items, const float *user_feat, int64_t num_user,
                                int32_t user_width, const float *item_feat, int64_t num_item, int32_t item_width, int64_t B,
                                float *out, int32_t *status, void *stream) {
  using namespace rs;
  RS_CHECK_ARG(B >= 0 && user_width >= 0 && item_width >= 0, RS_E_ARG, "rs_assemble_features: negative size");
  if (B == 0) return 0;
  RS_CHECK_ARG(users && items && out && status, RS_E_ARG, "rs_assemble_features: null ids/out/status");
  RS_CHECK_ARG((user_width == 0 || (user_feat && num_user > 0)) && (item_width == 0 || (item_feat && num_item > 0)), RS_E_ARG,
               "rs_assemble_features: missing side-feature table");
  const int64_t total = B * (2 + user_width + item_width);
  int64_t blocks = (total + 255) / 256;
  int64_t cap = (int64_t)num_sms() * 16;
  assemble_features_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, (cudaStream_t)stream>>>(
      users, items, user_feat, num_user, user_width, item_feat, num_item, item_width, B, out, status);
  RS_CHECK_LAUNCH();
  return 0;
}
