/*
 * recsys_b200.h -- C ABI of the B200 (sm_100a) embedding -> interaction -> sparse-update hot path.
 *
 * The reference (WardellZc/DeepLearningRecommendationSystem) is pure Python and has NO FFI layer; its
 * "plugin interface" for this path is the nn.Module / optimizer protocol used by trainer/trainer.py:23-40.
 * Each entry point below cites the reference call it replaces.  The Python host mirror
 * (deeplearningrecommendationsystem_b200/) binds these symbols with ctypes; INTEGRATION.md shows the stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - every data pointer is a DEVICE pointer owned by the caller (no allocation, no ownership transfer);
 *     structs themselves (rs_tables, rs_fields_io, ...) are HOST memory, read during the call;
 *   - all calls are asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return value: 0 on success, RS_E_* (< 0) on a bad argument, a positive cudaError_t on a launch
 *     failure; rs_last_error() gives a message; nothing throws across the boundary;
 *   - arithmetic is fp32, ids are int64, exactly as the reference's CPU path;
 *   - out-of-range ids never fault: the lookup is clamped and bit 0 of the optional device word
 *     `status` is set (the host mirror turns that into the reference's IndexError).
 */
#ifndef RECSYS_B200_H
#define RECSYS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RS_MAX_FIELDS 64
#define RS_CHUNK 64 /* sorted lookups summed sequentially by one lane group (segment-reduce granularity) */
#define RS_UNIT 512 /* sorted lookups per dynamically scheduled work unit of the streaming update kernel */

enum { RS_OK = 0, RS_E_ARG = -1, RS_E_SHAPE = -2, RS_E_WORKSPACE = -3, RS_E_UNSUPPORTED = -4 };

/* F embedding tables read by one lookup call; field f's table is base[f], shape (rows[f], width) fp32,
 * row-major.  A single concatenated table is the special case base[f] = weight + row_offset[f]*width. */
typedef struct rs_tables {
  int32_t num_fields;
  int32_t width;
  const float *base[RS_MAX_FIELDS];
  int64_t rows[RS_MAX_FIELDS];
} rs_tables;

/* Destination routing for rows that leave this GPU over NVLink peer memory: rows [start[k], start[k+1]) of the
 * logical output go to base[k] + (row0[k] + (r - start[k])) * width floats.  base[k] is a device pointer into rank k's
 * symmetric (peer-mapped) buffer, or into local memory for k == own rank.  n == 0 means "no routing". */
#define RS_MAX_RANKS 64
typedef struct rs_routes {
  int32_t n;
  int64_t start[RS_MAX_RANKS + 1];
  float *base[RS_MAX_RANKS];
  int64_t row0[RS_MAX_RANKS];
  /* Optional DEVICE-resident ranges (the host-sync-free sharded step: the split sizes only ever exist on the device).
   * When dyn_start != NULL the kernels read start[0..n] from dyn_start and row0[0..n-1] from dyn_row0 instead of the
   * host arrays above; a destination row index >= cap_rows (cap_rows > 0) is dropped, not stored. */
  const int64_t *dyn_start;
  const int64_t *dyn_row0;
  int64_t cap_rows;
  /* Own index among the n destinations (-1 = unknown).  When every rank pushes to the destinations in the same order
   * (rows are sorted owner-major), all of them hit destination 0 first, then 1, ...: an n-way incast on one NVLink ingress
   * at a time.  Knowing `self`, the kernels start their walk over the rows at self/n of the way through, so that at any
   * moment rank r is sending to rank (r + t) % n -- the classic all-to-all schedule.  Results do not depend on it. */
  int32_t self;
} rs_routes;

int rs_version(void);
const char *rs_last_error(void);

/* ---- gather: replaces nn.Embedding.forward (model/deepfm.py:45-46, model/mf.py:24-25, model/din.py:35-36).
 * out[b, f, :] = T.base[f][ids[b, f], :]   -- a pure copy, bit-exact.  ids (B, F) int64, out (B, F, width). */
int rs_gather_rows(const rs_tables *T, const int64_t *ids, int64_t B, float *out, int32_t *status, void *stream);
/* Fused gather + all-to-all for row-sharded tables: row i of the request list (local indices `idx`, grouped by
 * requesting rank) is copied from `table` straight into the requester's receive block through its peer-mapped
 * pointer (routes), i.e. the owner's gather kernel IS the "rows" all-to-all.  A cross-rank barrier must follow. */
int rs_gather_rows_peer(const float *table, int64_t rows, int32_t width, const int64_t *idx, int64_t m,
                        const rs_routes *routes, int32_t *status, void *stream);

/* ---- fused multi-field lookup + interaction forward.
 * Replaces the per-model python between the embedding calls and the MLP:
 *   FM sum-square second order          model/deepfm.py:71-77
 *   NFM bi-interaction pooling          model/nfm.py:58-62
 *   PNN inner products                  model/pnn.py:61-66
 *   field concat for the deep tower     model/deepfm.py:54, model/pnn.py:55, model/neuralcf.py:46
 *   MF dot / GMF Hadamard (F == 2)      model/mf.py:26, model/neuralcf.py:39
 * Source of the (B, F, D) field embeddings: `ids` (gather from T) or, when ids == NULL, the dense tensor
 * `dense_in` (already-materialised embeddings, used by the MovieLens feature-vector front end).
 * Any subset of the outputs may be requested (NULL = not wanted). */
typedef struct rs_fields_io {
  const int64_t *ids;     /* (B, F) or NULL */
  const float *dense_in;  /* (B, F, D) when ids == NULL */
  float *cross;           /* (B)      0.5 * sum_d[(sum_f e)^2 - sum_f e^2]                       */
  float *bi;              /* (B, D)   0.5 * [(sum_f e)^2 - sum_f e^2]  == sum_{i<j} e_i * e_j   */
  float *pairs;           /* (B, F(F-1)/2)  <e_i, e_j>, i<j in nested-loop order                 */
  float *concat;          /* (B, F*D) the gathered rows                                           */
  float *stash;           /* (B, F, D) S_b - e_bf : d cross / d e_bf, consumed by rs_segment_update */
  float *dot2;            /* (B)      <e_0, e_1>            (F == 2 only)                         */
  float *had2;            /* (B, D)   e_0 * e_1             (F == 2 only)                         */
} rs_fields_io;
int rs_fields_fwd(const rs_tables *T, const rs_fields_io *io, int64_t B, int32_t *status, void *stream);

/* Backward of the same interactions w.r.t. the field embeddings (autograd of the python listed above):
 *   dE[b,f,:] = g_cross[b]*(S_b - e_bf) + g_bi[b,:]*(S_b - e_bf) + sum_{j!=f} g_pairs[b,(f,j)]*e_bj
 *             + g_concat[b,f,:] + (F==2) g_dot2[b]*e_other + g_had2[b,:]*e_other
 * Any upstream gradient may be NULL.  dE (B, F, D) is the per-lookup row gradient that rs_segment_update
 * reduces over duplicate ids. */
typedef struct rs_fields_grad {
  const int64_t *ids;
  const float *dense_in;
  const float *g_cross, *g_bi, *g_pairs, *g_concat, *g_dot2, *g_had2;
  float *dE;
} rs_fields_grad;
int rs_fields_bwd(const rs_tables *T, const rs_fields_grad *g, int64_t B, void *stream);

/* ---- FFM: field-aware lookup + pairwise interaction  (model/ffm.py:46-82, generalised to F fields).
 * Table row of feature i = (F, D): slot j is v_{i,j}, feature i's vector toward field j.
 *   cross[b] = sum_{i<j} <v_{i,j}(b), v_{j,i}(b)>
 *   stash[b, i, j, :] = v_{j,i}(b) (0 on the diagonal) = d cross[b] / d v_{i,j}(b), the Jacobian row that
 *   rs_segment_update scales by dL/dcross[b]; pass NULL for inference.
 * Rows travel global->shared with cp.async.bulk (TMA bulk copy) through an mbarrier ring. */
int rs_ffm_fwd(const rs_tables *T /* width = F*D */, const int64_t *ids, int64_t B, int32_t D, float *cross,
               float *stash, int32_t *status, void *stream);
/* Row-sharded variant: fields whose bit is set in direct_mask are read straight from the owning rank's shard
 * (shard[g % world] + (g / world) * width, peer-mapped pointers) with ids[b, f] = GLOBAL row g; the other fields are read
 * from T as in rs_ffm_fwd (ids = row of T->base[f], typically the fetched block).  Same outputs. */
typedef struct rs_peer_tables {
  int32_t world;
  uint64_t direct_mask;
  const float *shard[RS_MAX_RANKS];
  int64_t total_rows; /* bound for the global rows of the direct fields */
  /* optional split stash: when stash_split != NULL the Jacobian rows of the fields in split_mask go to
   * stash_split (B, popcount(split_mask), F*D), field order preserved, and `stash` holds only the other fields'
   * rows (B, F - popcount, F*D) -- the replicated and the row-sharded tables of one model are reduced separately */
  uint64_t split_mask;
  float *stash_split;
} rs_peer_tables;
int rs_ffm_fwd_peer(const rs_tables *T /* width = F*D */, const int64_t *ids, int64_t B, int32_t D, const rs_peer_tables *PT,
                    float *cross, float *stash, int32_t *status, void *stream);
/* Dense small-F variant used by the MovieLens FFM module: Tin (B, F, NF, D), field_of[F] (host). */
int rs_ffm_dense_fwd(const float *Tin, int64_t B, int32_t F, int32_t NF, int32_t D, const int32_t *field_of,
                     float *cross, void *stream);
int rs_ffm_dense_bwd(const float *Tin, const float *g_cross, int64_t B, int32_t F, int32_t NF, int32_t D,
                     const int32_t *field_of, float *dT, void *stream);

/* ---- deterministic dedup: stable sort of the lookups by table row + segment boundaries.
 * Replaces the bookkeeping inside autograd's embedding_dense_backward (implicit at trainer/trainer.py:38).
 * (uniq, inverse, counts) equal torch.unique(keys, sorted=True, return_inverse=True, return_counts=True)
 * where keys[p] = row_offset[p % F] + ids[p]. */
typedef struct rs_segments {
  uint32_t *sorted_key;      /* [n]   global row of each lookup, ascending                        */
  int32_t *sorted_pos;       /* [n]   lookup index p = b*F+f; ascending inside a segment (stable) */
  int64_t *uniq;             /* [n]   first *n_uniq entries valid                                 */
  int32_t *inverse;          /* [n]   segment index of lookup p                                   */
  int32_t *counts;           /* [n]                                                               */
  int32_t *seg_start;        /* [n+1] start of each segment in the sorted order                   */
  int32_t *seg_first_chunk;  /* [n+1]                                                             */
  int32_t *chunk_start;      /* [n+1] segments cut into chunks of <= RS_CHUNK lookups             */
  int32_t *chunk_seg;        /* [n]                                                               */
  int32_t *multi_seg;        /* [n]   segments that span more than one chunk (any order)          */
  int32_t *lookup_desc;      /* [n*4] per sorted lookup: {pos, flags(1 first|2 last|4 single-chunk segment),
                                 global row, partial slot} -- the record the streaming update kernel reads */
  int32_t *work_counter;     /* [1]   dynamic work-unit counter of the streaming update kernel     */
  int32_t *unit_start;       /* [n/RS_UNIT + 2] first chunk start at or after u*RS_UNIT (work-unit boundaries) */
  float *scale_sorted;       /* [n]   scratch: per-sample scale permuted into sorted-lookup order   */
  int32_t *n_uniq;           /* [1] device scalar                                                 */
  int32_t *n_chunks;         /* [1] device scalar                                                 */
  int32_t *n_multi;          /* [1] device scalar                                                 */
  float *partial;            /* scratch for chunk partial sums, sized by rs_dedup_workspace_bytes */
  int64_t partial_floats;
} rs_segments;
int rs_dedup_workspace_bytes(int64_t n, int32_t max_width, size_t *bytes);
/* row_offset: HOST array of F int64 (NULL = all zero).  Fills `seg` with pointers carved from ws. */
int rs_dedup_sort(const int64_t *ids, int64_t n, int32_t F, const int64_t *row_offset, int64_t total_rows,
                  void *ws, size_t ws_bytes, rs_segments *seg, int32_t *status, void *stream);
/* Extended form used by the row-sharded step (no reference counterpart; SURVEY.md 8e):
 *   n_valid      DEVICE int32 (NULL = n): only the first *n_valid ids exist; the rest of the n-entry buffer is padding
 *                (a fixed-capacity receive list whose fill level is only known on the device).  Padding sorts last and
 *                produces no segment, chunk or work unit, so rs_segment_update over the same n touches valid rows only.
 *   shard_world  > 1: keys become owner-major, key = (g % shard_world) * shard_rows + g / shard_world for global row
 *                g = row_offset[p % F] + ids[p] -- one sort then yields the distinct rows grouped by owning rank. */
typedef struct rs_dedup_opts {
  const int32_t *n_valid;
  int32_t shard_world;
  int64_t shard_rows;
} rs_dedup_opts;
int rs_dedup_sort_ex(const int64_t *ids, int64_t n, int32_t F, const int64_t *row_offset, int64_t total_rows,
                     const rs_dedup_opts *opts, void *ws, size_t ws_bytes, rs_segments *seg, int32_t *status, void *stream);
/* Rename the rows of a finished sort to their rank among the distinct keys: uniq[g] := g and every lookup record
 * points at g.  The row-sharded step (no reference counterpart; SURVEY.md 8e) sorts the batch's GLOBAL rows once for
 * the exchange plan; the j-th distinct row is row j of the fetched block, so after this call the same segments drive
 * the per-row gradient reduce over the block -- no second sort. */
int rs_segments_relabel(const rs_segments *seg, int64_t n, void *stream);

/* ---- segment-reduce of duplicate rows fused with the row update.
 * Replaces embedding_dense_backward + optimizer.step() for embedding tables (trainer/trainer.py:38-39).
 * Gradient of lookup p (sample b = p / F):  G[p,:] = scale[b]*stash[p,:] + dense[p,:]   (either may be NULL)
 *   scale_width 1: per-sample scalar (dL/dcross); == width: per-sample vector (dL/dbi), only with F*W stash.
 * For every unique row r the G[p] of its lookups are summed in ascending p (chunks of RS_CHUNK, then the
 * chunk partials in order) -- deterministic -- and `mode` is applied to row r of `table` (global row index):
 *   RS_UPD_GRAD   dense_grad[r] = sum                     (table untouched; feeds stock torch optimisers)
 *   RS_UPD_SGD    w -= lr * (sum + wd*w)
 *   RS_UPD_ADAM   lazy row-wise Adam on (w, m[r], v[r]) with torch.optim.Adam's arithmetic */
enum { RS_UPD_GRAD = 0, RS_UPD_SGD = 1, RS_UPD_ADAM = 2 };
typedef struct rs_update {
  int32_t mode;
  int32_t width;
  int32_t F;
  int32_t scale_width;
  const float *stash, *scale, *dense;
  float *table;       /* (total_rows, width) */
  float *m, *v;       /* Adam moments, same shape */
  float *dense_grad;  /* RS_UPD_GRAD target, same shape, pre-zeroed by the caller */
  float lr, wd, beta1, beta2, eps;
  int32_t step;       /* 1-based */
  const rs_routes *grad_routes; /* RS_UPD_GRAD only, optional: write row r of the reduced gradient to a peer
                                   (routes) instead of dense_grad[r] -- segment-reduce fused with the gradient push */
  int32_t half_sm;    /* != 0: the streaming kernel takes one CTA and half of the shared memory per SM, so that a second
                         streaming update launched on another stream runs beside it (an NVLink-bound gradient push next to
                         an HBM-bound local reduce) */
} rs_update;
int rs_segment_update(const rs_segments *seg, int64_t n, const rs_update *u, void *stream);

/* ---- FFM training step WITHOUT the full Jacobian stash (autograd of model/ffm.py:61-82 + embedding_dense_backward +
 * optimizer.step(), trainer/trainer.py:38-39).  The gradient of table row (b, i) is dL/dcross[b] * [v_{j,i}(b)]_j, i.e.
 * slot i of the other rows of sample b, so it can be rebuilt from the (not yet updated) table instead of being written
 * out whole by rs_ffm_fwd.  Fields are split by `cold_mask` (bit f set = field f is a LARGE table):
 *   rs_ffm_fwd_train   forward; writes only the "cold-slice stash" cold_stash[b, i, c, :] = v_{cold_c, i}(b)
 *                      (B, F, nC, D), nC = popcount(cold_mask): the slices that live in rows of the large tables
 *                      (nC/F of a full stash; random 64-byte reads into a many-GB table are TLB-miss bound);
 *   rs_ffm_bwd_update  rows of cold fields looked up once in the batch are updated in place by the CTA that holds their
 *                      sample's tile; every other row is reduced in sorted order from gathered slices (small-field
 *                      slices straight from the table -- L2 resident --, cold ones from cold_stash), buffered, and
 *                      applied after every read is over.
 * Same per-element arithmetic, chunking and combine order as rs_ffm_fwd(stash) + rs_segment_update(stash, scale)
 * => identical bits.  `seg` = rs_dedup_sort of the same ids (partial scratch sized for width F*D); `u`: mode RS_UPD_SGD,
 * width = F*D, F, table = the concatenated table the T->base[f] point into, scale = dL/dcross (B), lr, wd; stash /
 * dense must be NULL.  The table must not have changed since the forward.  ws: rs_ffm_bwd_ws_bytes(n = B*F, B, width). */
int rs_ffm_fwd_train(const rs_tables *T /* width = F*D */, const int64_t *ids, int64_t B, int32_t D, uint64_t cold_mask,
                     float *cross, float *cold_stash, int32_t *status, void *stream);
int rs_ffm_bwd_ws_bytes(int64_t n, int64_t B, int32_t width, size_t *bytes);
int rs_ffm_bwd_update(const rs_tables *T /* width = F*D */, const int64_t *ids, int64_t B, int32_t D, uint64_t cold_mask,
                      const float *cold_stash, const rs_segments *seg, const rs_update *u, void *ws, size_t ws_bytes,
                      int32_t *status, void *stream);

/* ---- row-sharded tables: the exchange plan lives on the DEVICE (no reference counterpart; SURVEY.md 8e).
 * Global row g is owned by rank g % world at local index g / world.  Every rank owns two small symmetric (peer-mapped)
 * buffers: `req` (world slots of cap_req int32 local row indices, slot r written by requester r) and `ctl`
 * (RS_SHARD_CTL_WORDS int64 control words).  One step:
 *   rs_dedup_sort_ex(shard_world)   distinct rows of the local batch, grouped by owner
 *   rs_shard_post                   requester: writes its request list and counts straight into every owner's req/ctl
 *   -- cross-rank barrier --
 *   rs_shard_collect                owner: prefix of the counts, compact receive list, tells every requester where its
 *                                   gradients will go (ctl of the requester)
 *   rs_shard_serve                  owner: table rows -> the requesters' blocks over NVLink (TMA bulk copies for wide rows)
 *   -- barrier --  forward / backward on the fetched block  --
 *   rs_segment_update(RS_UPD_GRAD, grad_routes with dyn_start = ctl + RS_CTL_SEND_START, dyn_row0 = ctl + RS_CTL_G0_IN)
 *   -- barrier --
 *   rs_dedup_sort_ex(n_valid = m_total) + rs_segment_update on the received rows.
 * Nothing in this sequence reads a count on the host, so the whole step can be captured in a CUDA graph.
 * Bit 4 (16) of `status` is set when an owner is asked for more rows than cap_recv. */
#define RS_SHARD_CTL_WORDS 384
enum { RS_CTL_CNT_IN = 0, RS_CTL_BLK0_IN = 64, RS_CTL_G0_IN = 128, RS_CTL_SEND_START = 192, RS_CTL_RECV_START = 257, RS_CTL_M_TOTAL = 322 };
#define RS_MAX_DIRECT 8
typedef struct rs_shard {
  int32_t world, rank;
  int64_t rows_per_rank; /* R = ceil(total_rows / world) */
  int64_t cap_req;       /* ids per (requester, owner) slot; >= lookups per batch */
  int64_t cap_recv;      /* rows one owner can receive per step */
  int32_t *req[RS_MAX_RANKS];
  int64_t *ctl[RS_MAX_RANKS];
  /* "Direct" global-row ranges [direct_lo[k], direct_hi[k]): fields so large that a batch's lookups are (nearly) all
   * distinct, so fetching their rows into the block first saves nothing.  Their requests are flagged (recv_skip) and a
   * forward kernel that can read peer shards itself (rs_ffm_fwd_peer) pulls those rows straight over NVLink inside its
   * own TMA pipeline -- the transfer then overlaps the forward's HBM traffic instead of preceding it. */
  int32_t n_direct;
  int64_t direct_lo[RS_MAX_DIRECT], direct_hi[RS_MAX_DIRECT];
} rs_shard;
int rs_shard_post(const rs_shard *S, const rs_segments *seg, int64_t n, int32_t *status, void *stream);
/* recv_skip [cap_recv] (may be NULL when n_direct == 0): 1 for received requests that lie in a direct range. */
int rs_shard_collect(const rs_shard *S, int64_t *recv_local /* [cap_recv] */, uint8_t *recv_skip, int32_t *m_total /* device */,
                     int32_t *status, void *stream);
/* block[r]: base of rank r's receive block (cap_block_rows x width fp32), peer-mapped.  skip != NULL: rows flagged there
 * are not copied (their block slots stay untouched). */
int rs_shard_serve(const rs_shard *S, const float *table, int64_t rows, int32_t width, const int64_t *recv_local,
                   const uint8_t *skip, float *const *block, int64_t cap_block_rows, int32_t *status, void *stream);

/* Replicated small tables (SURVEY.md 8e: "small tables + all dense params: replicated; gradients all-reduced"): every rank
 * holds the same copy w[k] of the table and its own dense gradient g[k] (symmetric memory, peer-mapped pointers indexed
 * by rank; numel floats each).  Rank `rank` owns the rank-th slice of the elements: it adds the `world` gradient slices
 * in rank order, applies w -= lr * (sum + wd * w) to that slice and stores the result into every rank's copy -- the
 * reduce-scatter, the SGD step and the all-gather in one kernel; replicas stay bit-identical.  Cross-rank barriers must
 * precede (all g complete) and follow (before g or w are touched again) the call. */
int rs_replica_sgd(float *const *w, const float *const *g, int64_t numel, int32_t world, int32_t rank, float lr, float wd,
                   void *stream);
/* Replicated small tables with the LAZY row update (weight decay and/or Adam): only rows that some rank's batch touched
 * step, as in rs_segment_update; the others keep their bits (w, m and v).
 *   rs_mark_rows       touched[uniq[j]] = 1 for j < *seg->n_uniq (read on the device; `n` = the sort's lookup count only
 *                      sizes the grid).  touched: this rank's own uint8 array of `rows` flags in symmetric memory, zeroed
 *                      by the caller on the stream beforehand.  Ranks never write each other's flags.
 *   rs_replica_update  rank `rank` owns the float4 slice [lo4, hi4) of n4 = numel / 4, per = ceil(n4 / world),
 *                      lo4 = min(rank * per, n4), hi4 = min(lo4 + per, n4) -- rs_replica_sgd's slices.  For each float4 i
 *                      of row i * 4 / width (width % 4 == 0, so a float4 never straddles rows; a slice may split a row) it
 *                      ORs the `world` flags touched[r][row]; an untouched element is skipped (no load, no store).
 *                      Otherwise the `world` gradients g[r] are added in rank order (rs_replica_sgd's sum), u->mode
 *                      (RS_UPD_SGD or RS_UPD_ADAM; others are refused) is applied with rs_segment_update's arithmetic and
 *                      bias correction (u->lr, wd, beta1, beta2, eps, step), and w is stored into every replica.  The
 *                      flags decide, not the gradient: a touched row whose summed gradient is exactly zero still steps.
 *                      Adam's moments are NOT replicated: u->m / u->v point at this rank's slice only ((hi4 - lo4) * 4
 *                      floats, element 0 = element lo4 * 4 of the table); u->width = row width.
 * Barriers: every rank's g and flags must be complete before any rank calls rs_replica_update (the barrier after the
 * gradient reduce), and a cross-rank barrier must follow it before any rank zeroes its flags or gradient, or touches w,
 * again. */
int rs_mark_rows(const rs_segments *seg, int64_t n, uint8_t *touched, int64_t rows, int32_t *status, void *stream);
int rs_replica_update(float *const *w, const float *const *g, const uint8_t *const *touched, int64_t numel, int32_t world,
                      int32_t rank, const rs_update *u, void *stream);

/* Fused DENSE Adam sweep with torch.optim.Adam's exact arithmetic order ("reference-Adam" mode for the
 * MovieLens-sized tables; scripts/deepfm.py:55). */
int rs_adam_dense(float *p, const float *g, float *m, float *v, int64_t numel, float lr, float wd, float beta1,
                  float beta2, float eps, int32_t step, void *stream);

/* ---- MovieLens feature-vector front end (x (B,45) f32, data/reader.py:98-101 column order).
 * Each output "slot" t is described by (col, ncols, kind): kind 0 = id column -> row gather
 * (model/deepfm.py:45-46), 1 = one-/multi-hot bag -> sum_k x[b,col+k]*W_t[k,:] (the matmul at
 * model/deepfm.py:47-51), 2 = scalar broadcast over D (AFM's age, model/afm.py:45,54; no table). */
typedef struct rs_xslots {
  int32_t num_slots, width, xcols;
  int32_t col[RS_MAX_FIELDS], ncols[RS_MAX_FIELDS], kind[RS_MAX_FIELDS];
  const float *table[RS_MAX_FIELDS];
  int64_t rows[RS_MAX_FIELDS];
} rs_xslots;
int rs_xembed_fwd(const rs_xslots *S, const float *x, int64_t B, float *E /* (B, slots, width) */,
                  int32_t *status, void *stream);
/* bag-table gradient: dW_t[k,:] = sum_b x[b,col+k]*dE[b,t,:], two-pass fixed-order reduction.
 * dW[t] points at a (ncols[t], width) buffer (NULL for non-bag slots); ws holds the block partials. */
int rs_xembed_bag_bwd(const rs_xslots *S, const float *x, const float *dE, int64_t B, float *const *dW,
                      float *ws, size_t ws_bytes, void *stream);
int rs_xembed_bag_ws_bytes(const rs_xslots *S, int64_t B, size_t *bytes);
/* float-encoded id column -> int64 (x[:,c].long(), model/deepfm.py:45) */
int rs_xcol_to_ids(const float *x, int64_t B, int32_t xcols, int32_t col, int64_t *ids, void *stream);

/* ---- AFM attention pooling over the pairwise Hadamard products (model/afm.py:55-65).
 *   P_p = e_i*e_j (i<j), s_p = h.relu(P_p W + b), w = softmax_p(s), pooled = sum_p w_p P_p
 * E (B, F, D) dense field embeddings, W (D, A), b (A), h (A).  The (B, P, D) pair tensor is never materialised.
 * Forward saves the softmax weights attw (B, P) for the backward.  Backward returns dE and PER-WARP partial sums of
 * dW (parts, D, A), db (parts, A), dh (parts, A) -- add them over `parts` (= rs_afm_num_parts) in index order. */
int rs_afm_num_parts(int64_t B, int32_t F, int32_t D, int32_t A, int32_t *parts);
int rs_afm_fwd(const float *E, int64_t B, int32_t F, int32_t D, int32_t A, const float *W, const float *bvec,
               const float *h, float *pooled /* (B,D) */, float *attw /* (B,P) or NULL */, void *stream);
int rs_afm_bwd(const float *E, int64_t B, int32_t F, int32_t D, int32_t A, const float *W, const float *bvec,
               const float *h, const float *attw, const float *g_pooled, float *dE, float *dW_part, float *db_part,
               float *dh_part, int32_t num_parts, void *stream);

/* Tensor-core backward of the AFM pooling (afm_tc.cu) for the shapes its forward serves (D in {16, 32}, A in {32, 64,
 * 128}, >= 128 pairs, B >= 2 x SMs).  rs_afm_bwd_tc_plan returns num_parts == 0 when the shape is served by rs_afm_bwd
 * instead.  dE (B, F, D) is complete; the parameter gradients come back as per-warpgroup partials U_part (parts, D, A)
 * and m1_part (parts, A), to be added in index order:  with U = sum U_part, m1 = sum m1_part,
 *   dW = U * h[a],   db = h * m1,   dh[a] = sum_d W[d][a] U[d][a] + b[a] m1[a]. */
int rs_afm_bwd_tc_plan(int64_t B, int32_t F, int32_t D, int32_t A, int32_t *num_parts, size_t *ws_bytes);
int rs_afm_bwd_tc(const float *E, int64_t B, int32_t F, int32_t D, int32_t A, const float *W, const float *bvec,
                  const float *h, const float *attw, const float *g_pooled, float *dE, float *U_part, float *m1_part,
                  int32_t num_parts, void *ws, size_t ws_bytes, void *stream);

/* ---- DIN target attention (model/din.py:39-47; model/dien.py:27-37 with pool == 0), forward and backward.
 * rows (B, L+1, D): the L gathered history rows followed by the target row (the layout rs_gather_rows produces for
 * ids = [hist | target]).  Attention unit 3D -> H1 -> H2 -> 1 with ReLU (torch Linear layout (out, in)), softmax over
 * L without mask or scaling.  pool != 0: out (B, D) = sum_l w_l h_l;  pool == 0: out (B, L, D) = w_l h_l.
 * The concat [h, h-t, t] is never built: W0 z = (Wa+Wb) h + (Wc-Wb) t.  Built for D in {16,32,64} and
 * (H1,H2) in {(128,64),(64,32)}.
 * Backward recomputes the activations; d_rows (B, L+1, D) is the gradient THROUGH the attention (add the direct uses
 * of the rows outside).  Weight gradients come back as per-CTA partials (num_parts = rs_din_num_parts(B)), to be
 * added in index order:  dW0 = [dWab | dWab - dWt | dWt]  with dWab, dWt (parts, H1, D);  dW1 (parts, H2, H1);
 * db0 (parts, H1); db1 (parts, H2); dW2 (parts, H2); db2 (parts). */
typedef struct rs_din_weights {
  const float *W0, *b0, *W1, *b1, *W2, *b2;
  int32_t H1, H2;
} rs_din_weights;
int rs_din_num_parts(int64_t B, int32_t *parts);
int rs_din_fwd(const float *rows, int64_t B, int32_t L, int32_t D, const rs_din_weights *w, int32_t pool, float *out,
               float *attw /* (B, L) or NULL */, void *stream);
/* Same contract as rs_din_fwd with the two hidden layers on the tcgen05 tensor cores (3xTF32, fp32 accumulation in
 * tensor memory): 128 (b, l) rows per tile, layer-0 epilogue feeds layer 1's operand through shared memory, scores
 * then softmax + weighted sum.  ws: rs_din_fwd_tc_ws_bytes (per-sample target bias (B, H1) + scores (B, L)).
 * Built for D in {16,32,64}, H1 in {64,128}, H2 in {32,64}. */
int rs_din_fwd_tc_ws_bytes(int64_t B, int32_t L, int32_t D, int32_t H1, int32_t H2, size_t *bytes);
int rs_din_fwd_tc(const float *rows, int64_t B, int32_t L, int32_t D, const rs_din_weights *w, int32_t pool, float *out,
                  float *attw /* (B, L) or NULL */, float *act0 /* (B*L, H1) or NULL */, float *act1 /* (B*L, H2) or NULL */,
                  void *ws, size_t ws_bytes, void *stream);
/* Backward of rs_din_fwd_tc from its stashes (attw and the two ReLU outputs act0, act1), data-gradient chain on the
 * tensor cores:  ds = softmax backward (scratch, (B, L));  dz1 = ds w2 [act1 > 0] (B*L, H2);  dz0 = (dz1 W1) [act0 > 0]
 * written as (B, L+1, H1) with a zero row in the target slot;  d_rows[b, l<L] = dz0 (Wa+Wb) + w_l g  (the target row
 * d_rows[b, L] is NOT written).  The weight gradients are reductions over all rows that the caller forms from the
 * outputs with rs_gemm_tn_3xtf32 and small sums:
 *   dW1 = dz1^T act0,  dWab = dz0^T rows,  db1 = sum dz1,  dW2 = ds^T act1,  db2 = sum ds,
 *   dtb = sum_l dz0 (B, H1),  db0 = sum_b dtb,  dWt = dtb^T t,  d_rows[b, L] = dtb (Wc - Wb),
 *   dW0 = [dWab | dWab - dWt | dWt]. */
int rs_din_bwd_tc(const float *rows, int64_t B, int32_t L, int32_t D, const rs_din_weights *w, int32_t pool,
                  const float *g_out, const float *attw, const float *act0, const float *act1, float *d_rows, float *dz0,
                  float *dz1, float *ds, void *stream);
int rs_din_bwd(const float *rows, int64_t B, int32_t L, int32_t D, const rs_din_weights *w, int32_t pool,
               const float *g_out, float *d_rows, float *dWab_part, float *dWt_part, float *dW1_part, float *db0_part,
               float *db1_part, float *dW2_part, float *db2_part, int32_t num_parts, void *stream);

/* ---- GRU recurrence (nn.GRU(D, H, batch_first=True), one layer, h0 = 0, gate order r,z,n; model/dien.py:47,61).
 * The input projection gi = x.W_ih^T + b_ih (B, L, 3H) is a plain library GEMM done by the caller; rs_gru_fwd runs
 * the L sequential steps (W_hh register-resident, BT batch rows per CTA): h_all (B, L, H) and, for BPTT,
 * gates (B, L, 4H) = r | z | n | (W_hn.h + b_hn)  (NULL for inference).  H in {8,16,32,64}.
 * rs_gru_bwd walks t = L-1..0 from g_h_all (B, L, H) and/or g_h_last (B, H) and emits d_gi and d_gh (B, L, 3H);
 * dW_ih = d_gi^T.x, dW_hh = d_gh^T.h_prev, dx = d_gi.W_ih and the bias sums are plain GEMMs/reductions on them. */
int rs_gru_fwd(const float *gi, int64_t B, int32_t L, int32_t H, const float *w_hh, const float *b_hh, float *h_all,
               float *gates, void *stream);
int rs_gru_bwd(const float *w_hh, const float *h_all, const float *gates, const float *g_h_all, const float *g_h_last,
               int64_t B, int32_t L, int32_t H, float *d_gi, float *d_gh, void *stream);

/* ---- C (M, N) = A^T B for row-major A (K, M), B (K, N): PNN "out" mode's batch-collapsed outer product
 * p = S^T S, S = sum_f e_f (model/pnn.py:69-72), on tcgen05 tensor cores with a 3xTF32 operand split (hi/lo) and fp32
 * accumulation in tensor memory, so the result stays within the path's 1e-5 bar.  M <= 128, N <= 256. */
int rs_gemm_tn_ws_bytes(int64_t K, int32_t M, int32_t N, size_t *bytes);
int rs_gemm_tn_3xtf32(const float *A, const float *B, int64_t K, int32_t M, int32_t N, float *C, float *ws,
                      size_t ws_bytes, void *stream);

/* C (M, N) = epilogue(A B^T) on tcgen05 (3xTF32): the DIN / DIEN attention-unit layers over all B*L rows
 * (model/din.py:14-20,43).  A (M, K): row r at A + (r / a_group)*a_group_stride + (r % a_group)*lda when a_group > 0
 * (rows of a (B, L+1, D) gather viewed as B*L history rows), else A + r*lda.  B (N, K) in torch Linear layout, kept
 * resident in shared memory (N <= 256, N*K bounded by shared memory).  Epilogue, in order: + bias[n],
 * + rowbias[r / rb_group][n], ReLU, zero where mask[r*ldm + n] <= 0. */
typedef struct rs_gemm_nt {
  const float *A, *B, *bias, *rowbias, *mask;
  float *C;
  int64_t M, lda, a_group, a_group_stride, ldb, rb_group, ldm, ldc;
  int32_t K, N, relu;
} rs_gemm_nt;
int rs_gemm_nt_3xtf32(const rs_gemm_nt *g, void *stream);

/* ---- sigmoid + BCELoss(mean) forward/backward in one pass (model/*: torch.sigmoid; scripts/deepfm.py:54).
 * pred = sigmoid(logit); loss_sum += sum(-[y*max(log p,-100)+(1-y)*max(log(1-p),-100)]);
 * g_logit follows autograd's op sequence ((p-y)/max(p(1-p),1e-12)/B * p(1-p)), i.e. (p-y)/B except where p
 * saturates.  loss_mean is a device scalar produced by a fixed-order two-pass reduce. */
int rs_sigmoid_bce(const float *logit, const float *y, int64_t B, float *pred, float *g_logit, float *loss_mean,
                   float *ws /* >= 1024 floats */, void *stream);
/* Same with the models' last step folded in: logit[b] = cross[b] + *bias (bias: device scalar or NULL), and
 * *g_sum = sum_b g_logit[b] (the bias gradient; NULL = not wanted), reduced in the same fixed order as the loss.
 * ws >= 2048 floats. */
int rs_sigmoid_bce_bias(const float *cross, const float *bias, const float *y, int64_t B, float *pred, float *g_logit,
                        float *loss_mean, float *g_sum, float *ws /* >= 2048 floats */, void *stream);

/* ---- catalogue ranking: the per-user `torch.topk(scores, k, dim=0)` of every recommendation() method
 * (model/deepfm.py:85-95, model/din.py:55-66, model/neuralcf.py:61-72, model/pnn.py:133-143 ...), all users in one launch.
 * Segment s covers scores[seg_start[s] .. seg_start[s+1]) (seg_start == NULL: uniform segments of max_len).
 * out_idx[s*k + r] = position inside segment s of its r-th largest score (descending; ties: lower position first;
 * NaN ranks highest, as torch.topk); out_val (optional) the scores in that order.  max_len is an upper bound of the
 * segment lengths (sizes the shared-memory slot buffer; up to 16384 in one pass, longer segments are streamed and then
 * need k <= 8192).  status |= 2 when a segment is shorter than k (its row is filled with -1), |= 4 when a segment
 * exceeded max_len and could not be finished. */
int rs_rank_segments(const float *scores, const int64_t *seg_start, int64_t num_segments, int64_t max_len, int32_t k,
                     int64_t *out_idx, float *out_val, int32_t *status, void *stream);

/* ---- fused MF scoring + ranking (model/mf.py:28-35: `U @ V^T` then topk over items): scores never reach HBM.
 * user_rows (num_users, width), item_rows (num_items, width) row-major fp32; out_* as rs_rank_segments with
 * uniform segments of num_items.  Each score is a fixed-order fp32 dot product.  For a small k over a large catalogue
 * (k <= 512, >= 64 users) a tiled kernel scores 8 users per CTA against a transposed copy of the item table held in
 * the caller's workspace (rs_mf_rank_ws_bytes; 0 when that path does not apply). */
int rs_mf_rank_ws_bytes(int64_t num_users, int64_t num_items, int32_t width, int32_t k, size_t *bytes);
int rs_mf_rank(const float *user_rows, const float *item_rows, int64_t num_users, int64_t num_items, int32_t width, int32_t k,
               int64_t *out_idx, float *out_val, int32_t *status, void *ws, size_t ws_bytes, void *stream);

/* ---- OPTIONAL device-side negative sampling (sampler/sampler.py:16-27: per user, num_negatives uniform items,
 * redrawn while (user, item) is an observed pair).  NOT the reference's python-`random` stream (that stays on the host,
 * sampler.Sampler); the stream is Philox4x32-10 with key = seed and counter = (sample index lo, hi, attempt block,
 * epoch), item = (r * num_item) >> 32, four attempts per block, first accepted wins -- restated bit for bit in
 * oracle/sampling.py.  excluded_keys: ascending int64 user * num_item + item.  out_* hold num_user * num_negatives
 * entries, user-major (the reference's order).  status |= 8 if a slot found no free item in 65536 attempts. */
int rs_sample_negatives(const int64_t *excluded_keys, int64_t num_excluded, int64_t num_user, int64_t num_item,
                        int32_t num_negatives, uint64_t seed, uint32_t epoch, int64_t *out_users, int64_t *out_items,
                        int32_t *status, void *stream);

/* ---- feature-matrix assembly (data/reader.py:98-101, the two pd.merge calls): out (B, 2 + user_width + item_width)
 * fp32 rows [user, item, user_feat[user, :], item_feat[item, :]].  status |= 1 on an out-of-range id. */
int rs_assemble_features(const int64_t *users, const int64_t *items, const float *user_feat, int64_t num_user,
                         int32_t user_width, const float *item_feat, int64_t num_item, int32_t item_width, int64_t B,
                         float *out, int32_t *status, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* RECSYS_B200_H */
