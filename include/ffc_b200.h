/*
 * ffc_b200.h -- C ABI of libffc_b200.so: the B200-native FFC classification head.
 *
 * The reference (sqnkkang/Very-Large-Scale-Face-Recognition) has no FFI: its hot path is two
 * Python classes, `LRU` (lru.py:21-255) and `FFC` (ffc.py:10-267).  This header is the boundary a
 * maintainer binds with ctypes (see INTEGRATION.md); every entry point names the reference code it
 * replaces.  Conventions:
 *   - plain C: pointers + sizes only, no C++/torch types; all `*_dev` pointers are CUDA device
 *     pointers owned by the caller; `stream` is a cudaStream_t passed as void*.
 *   - every function returns 0 on success, non-zero on error; ffc_last_error() gives the text.
 *   - nothing synchronises the stream unless stated ("host-sync").  Not thread-safe per handle.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails.
 *
 * Slots, rows and labels are int32 on the device (the reference uses Python ints / int64 tensors;
 * the Python mirror converts at the boundary).  Keys (identity labels) are int64; the two values
 * INT64_MIN and INT64_MIN+1 are reserved as hash-table sentinels and are rejected.
 */
#ifndef FFC_B200_H_
#define FFC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FFC_OK 0
#define FFC_ERR_INVALID 1
#define FFC_ERR_CUDA 2
#define FFC_ERR_STATE 3

#define FFC_LOSS_AM 0  /* ffc.py:73-94  CosFace / additive margin */
#define FFC_LOSS_ARC 1 /* ffc.py:95-115 ArcFace */
#define FFC_LOSS_SV 2  /* ffc.py:116-138 SV-softmax variant (mask_svfc = 1.2, ffc.py:47) */

#define FFC_PREC_BF16 0 /* tcgen05 bf16 tensor-core sweep (fp32 accumulate in TMEM)            */
#define FFC_PREC_FP32 1 /* check mode: fp32 inputs, fp64 accumulate, SIMT, no tensor cores     */

#define FFC_LRU_MAX_BATCH 1024 /* keys the single resolve CTA replays per chunk of a batch */
#define FFC_LRU_MAX_KEYS 65536 /* keys per ffc_lru_assign call (one launch pair; callers split larger batches) */
#define FFC_TOPK_MAX 10        /* ffc.py:48 hard_neg <= 10 */

const char* ffc_last_error(void);
/* library / build info: returns e.g. "ffc_b200 0.1 sm_100a" */
const char* ffc_version(void);

/* ------------------------------------------------------------------------------------------------
 * LRU id -> slot cache on the device (replaces lru.py:21-255 and the bookkeeping loop
 * ffc.py:162-177 / ffc.py:214-235).
 * State: open-addressing hash table key->slot (32-cell windows probed by one warp), slot_key[],
 * last_pos[] and a log-structured recency ring (one record per access; a record is live iff
 * last_pos[slot] == its ring position), cur_idx, an undo journal.
 * ---------------------------------------------------------------------------------------------- */
typedef struct ffc_lru ffc_lru_t;

/* lru.py:27-40 LRU.__init__(capacity).  journal_capacity: max outstanding journaled accesses
 * (try_get without rollback); 0 -> default 65536. */
int ffc_lru_create(int64_t capacity, int64_t journal_capacity, ffc_lru_t** out);
int ffc_lru_destroy(ffc_lru_t* h);
/* lru.py:132-141 clear(); unlike the reference it also resets cur_idx (the reference's clear()
 * leaves the object unusable, SURVEY.md 8(a) a6). */
int ffc_lru_clear(ffc_lru_t* h, void* stream);

/* B sequential accesses, in order, with the FFC bookkeeping folded in:
 *   journal == 0: lru.py:44-89  get()      for each key   (ffc.py:166-177)
 *   journal != 0: lru.py:157-204 try_get() for each key   (ffc.py:219-235), undo with ffc_lru_undo
 * Per position i:  cols_out[i] = slot;  rows_out[i] = 0 for a miss (and qpos[slot] = 1), or the
 * slot's qpos for a hit (then qpos[slot] ^= 1)              (ffc.py:167-177);
 * hit_out[i] = 1 for a hit.  Slots that were hit at least once are appended to ones_list_dev /
 * *n_ones_dev (a set: each slot once) and their bit is set in cmask_dev (bit s of word s/32) --
 * ffc.py:165,176 `ones_idx`.  qpos_dev (uint8[capacity]) is ffc.py:41-43 queue_position_dict; pass
 * NULL for a plain LRU (rows_out is then 0 for misses and 1 for hits... unspecified; pass NULL too).
 * Any of rows_out, hit_out, ones_list_dev, n_ones_dev, cmask_dev may be NULL.
 * 1 <= n <= FFC_LRU_MAX_KEYS: one lookup launch + one resolve launch whatever n is (the resolve CTA walks the batch in chunks
 * of FFC_LRU_MAX_BATCH keys); ring / table space for all n accesses is reserved before the first one.  n_ones_dev is
 * accumulated (caller zeroes it).
 * n_dev (optional device scalar) / n_base: when the number of keys is only known on the device (a rank's
 * share of an all-gathered batch), the call processes keys [0, clamp(*n_dev - n_base, 0, n)) and leaves the
 * outputs of the remaining positions untouched (the resolve CTA stops after the last non-empty chunk); pass NULL, 0 otherwise. */
int ffc_lru_assign(ffc_lru_t* h, const int64_t* keys_dev, int n, int journal, uint8_t* qpos_dev,
                   int32_t* rows_out, int32_t* cols_out, uint8_t* hit_out, int32_t* ones_list_dev,
                   int32_t* n_ones_dev, uint32_t* cmask_dev, const int32_t* n_dev, int n_base, void* stream);

/* lru.py:147-151 view() / lru.py:145-146 __contains__ for n keys: slot or -1, recency untouched
 * (ffc.py:189-194 / 242-246 probe labels).  Any n >= 1. */
int ffc_lru_view(ffc_lru_t* h, const int64_t* keys_dev, int n, int32_t* slots_out, void* stream);

/* lru.py:252-255 rollback_steps(steps): undo the newest `steps` journaled accesses (clamped to the
 * journal length, like the reference) including their qpos changes (ffc.py:256-257); steps < 0 undoes
 * everything outstanding. */
int ffc_lru_undo(ffc_lru_t* h, int64_t steps, uint8_t* qpos_dev, void* stream);

/* Bounded maintenance between passes (ring compaction, hash-table rebuild) when the host-side
 * conservative counters say so; never changes observable state. */
int ffc_lru_maintain(ffc_lru_t* h, void* stream);

/* host-sync: number of resident keys (== cur_idx) and outstanding journal length */
int ffc_lru_size(ffc_lru_t* h, int64_t* cur_idx_out, int64_t* journal_len_out, void* stream);
/* host-sync: lru.py:102-108 state_dict(): (key, slot) pairs from most to least recently used, into
 * HOST arrays of at least `capacity` entries; *n_out = count. */
int ffc_lru_export(ffc_lru_t* h, int64_t* keys_host, int32_t* slots_host, int64_t* n_out, void* stream);
/* host-sync: lru.py:113-128 restore(kvs): requires an empty cache (cur_idx == 0), n <= capacity,
 * distinct keys and distinct slots in [0, capacity). pairs are most- to least-recent. */
int ffc_lru_import(ffc_lru_t* h, const int64_t* keys_host, const int32_t* slots_host, int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Prototype queue scatter (replaces ffc.py:179-182, 237-241, 255).
 * queue_f32_dev: [2, Q, D] fp32 (the reference's `queue` buffer, checkpoint contract 'fc').
 * queue_bf16_dev: [2, Q, D] bf16 mirror read by the tensor-core sweep (may be NULL).
 * For each i with cols[i] >= 0: queue[rows[i], cols[i], :] = g[i, :]; a repeated (row, col) pair resolves to the LAST
 * occurrence (the reference's serial CPU behaviour; undefined on its CUDA path).
 * undo_f32_dev ([B, D] fp32, may be NULL): receives the previous fp32 row of every winning write so
 * that ffc_queue_restore can put it back (ffc.py:240 `old_tensor`, ffc.py:255).
 * ---------------------------------------------------------------------------------------------- */
int ffc_queue_scatter(float* queue_f32_dev, void* queue_bf16_dev, const int32_t* rows_dev,
                      const int32_t* cols_dev, const float* g_dev, int B, int64_t Q, int D,
                      float* undo_f32_dev, void* stream);
/* as ffc_queue_scatter with g[src_row[i], :] as the source row of position i (the sharded head scatters straight out of the
 * all-gathered embeddings) */
int ffc_queue_scatter_indexed(float* queue_f32_dev, void* queue_bf16_dev, const int32_t* rows_dev,
                              const int32_t* cols_dev, const float* g_dev, const int32_t* src_row_dev, int B,
                              int64_t Q, int D, float* undo_f32_dev, void* stream);
/* Sharded head: stable partition of n gathered gallery keys into (keys owned by `rank` under key mod n_ranks, the rest);
 * keys_out / order_out [n] (order_out[j] = source position), n_mine_out device scalar. */
int ffc_route_keys(const int64_t* keys_dev, int n, int n_ranks, int rank, int64_t* keys_out_dev,
                   int32_t* order_out_dev, int32_t* n_mine_out_dev, void* stream);
/* Cross-rank barrier on the stream (one tiny launch): tells every peer "what this rank stored into your buffers before this call is out"
 * (system-scope fence, release store of `epoch` into word my_rank of the peer's flag array) and waits until every peer has said so to this
 * rank.  flag_ptrs_dev[r] = rank r's peer-mapped array of n_ranks int32 words (zero-initialised; epochs only grow).  A wait longer than
 * 5 s raises *err_flag_dev and goes on (no hang). */
int ffc_peer_barrier(int32_t* const* flag_ptrs_dev, int my_rank, int n_ranks, int32_t epoch, int32_t* err_flag_dev, void* stream);

/* as ffc_queue_scatter_indexed, and every winning write also records in overlay_map_dev (int32 [2, Q], -1 = no entry; NULL = off)
 * where the content this (row, slot) had during the CURRENT pass's sweep stays available once later kernels have rewritten the row:
 *   overlay_table 0 (a rollback pass's enqueue): map = src_row[i]          -- the row is g[src_row[i]] until ffc_queue_restore
 *   overlay_table 1 (the commit pass that follows): map = 2^30 | i          -- undo[i] keeps what was there before; entries a table-0
 *                                                                             mark already holds are left alone (needs undo_f32_dev)
 * ffc_head_finalize_gathered_ex reads through the map; ffc_overlay_clear resets the entries of a pass's (rows, cols) list. */
int ffc_queue_scatter_overlay(float* queue_f32_dev, void* queue_bf16_dev, const int32_t* rows_dev,
                              const int32_t* cols_dev, const float* g_dev, const int32_t* src_row_dev, int B,
                              int64_t Q, int D, float* undo_f32_dev, int32_t* overlay_map_dev, int overlay_table,
                              void* stream);
int ffc_overlay_clear(int32_t* overlay_map_dev, const int32_t* rows_dev, const int32_t* cols_dev, int n, int64_t Q,
                      void* stream);
/* out[e] = slabs[e] + slabs[slab_stride + e] + ... (n_slabs terms, in that order), e < n: the local half of the reduce-scatter
 * that ffc_head_finalize_gathered_ex starts with its peer stores.  n and slab_stride multiples of 4. */
int ffc_sum_slabs(const float* slabs_dev, int n_slabs, int64_t slab_stride, int64_t n, float* out_dev, void* stream);
/* ffc_sum_slabs behind a barrier across the ranks, in one launch (the second half of the reduce-scatter that the peers' finalize
 * kernels started with their stores into this rank's staging buffer).  flag_ptrs_dev: device array of n_ranks pointers, entry r =
 * rank r's flag words (int32[n_ranks], peer-mapped, zero before the first step); epoch: the step number, growing by one per call on
 * every rank.  The kernel publishes `epoch` in every peer's flag word for this rank, waits until its own words have reached `epoch`,
 * then sums.  *err_flag_dev is set to 1 if the wait exceeds 5 s (no hang; the sums are then meaningless). */
int ffc_sum_slabs_barrier(const float* slabs_dev, int n_slabs, int64_t slab_stride, int64_t n, float* out_dev,
                          int32_t* const* flag_ptrs_dev, int my_rank, int n_ranks, int32_t epoch, int32_t* err_flag_dev,
                          void* stream);
int ffc_queue_restore(float* queue_f32_dev, void* queue_bf16_dev, const int32_t* rows_dev,
                      const int32_t* cols_dev, const float* undo_f32_dev, int B, int64_t Q, int D,
                      void* stream);
/* ffc_queue_restore for a PACKED list: the live positions (cols >= 0) come first, everything after the first padded position is
 * padded too -- what ffc_route_keys + ffc_lru_assign(n_dev) produce for a rank of the sharded head (its own keys compacted to the
 * front of the R*B gathered positions).  The duplicate scans stop at the first padded position.  ffc_queue_scatter_indexed /
 * ffc_queue_scatter_overlay make the same assumption about their lists. */
int ffc_queue_restore_packed(float* queue_f32_dev, void* queue_bf16_dev, const int32_t* rows_dev,
                             const int32_t* cols_dev, const float* undo_f32_dev, int B, int64_t Q, int D,
                             void* stream);
/* ------------------------------------------------------------------------------------------------
 * Gallery-network EMA (replaces ffc.py:139-145 _momentum_update_gallery), SURVEY 8(f) rank 1.
 * One launch over all parameter tensors: the caller splits every fp32 tensor into chunks of at most
 * ffc_ema_chunk_elems() elements and passes the chunk table (device memory).  g = g*m + p*one_minus_m with the
 * reference's rounding (two fp32 multiplies, one add, no FMA): bit-identical to the eager expression.
 * ---------------------------------------------------------------------------------------------- */
typedef struct ffc_ema_chunk {
  float* gallery;       /* updated in place */
  const float* probe;
  int32_t n;            /* elements in this chunk (<= ffc_ema_chunk_elems()) */
  int32_t pad;
} ffc_ema_chunk;
int ffc_ema_chunk_elems(void);
int ffc_ema_update(const ffc_ema_chunk* table_dev, int n_chunks, float m, float one_minus_m, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Backbone tail -> head hand-off, SURVEY 8(f) rank 3 (replaces the last two operations of every reference backbone:
 * `F.normalize(self.features(x))`, features = nn.BatchNorm1d(feat_dim, eps=1e-05) -- resnet_arcface.py:99,151,
 * resnet_std.py:201-202; plain `F.normalize(x)` in mobilefacenet_def.py:113-114 -- and their autograd backward).
 * The unit-norm fp32 rows the head consumes (ffc_head_pass.p_f32, ffc_queue_scatter's g) are written with a row stride,
 * so they can land directly in a packed staging buffer (the sharded head's all-gather input).
 * ---------------------------------------------------------------------------------------------- */
#define FFC_TAIL_NORMALIZE 0 /* p = x / max(||x||_2, 1e-12)                                       */
#define FFC_TAIL_BN_EVAL 1   /* BatchNorm1d with the running statistics (module.eval()), then normalise  */
#define FFC_TAIL_BN_TRAIN 2  /* BatchNorm1d with batch statistics (module.train()): running_mean / running_var are
                                updated as torch does (momentum, unbiased variance), then normalise      */

typedef struct ffc_tail_args {
  const float* x;        /* [n_rows, feat_dim] fp32, contiguous: the backbone's last linear output; must not alias p */
  float* p;              /* [n_rows] rows of feat_dim floats, p_stride floats apart: unit-norm output (input of backward) */
  int64_t p_stride;
  float* inv_norm;       /* [n_rows]: 1 / max(||y||, 1e-12), written by forward, read by backward */
  int32_t n_rows;
  int32_t feat_dim;
  int32_t mode;          /* FFC_TAIL_* */
  float eps;             /* BatchNorm1d eps (1e-05 in the reference) */
  float momentum;        /* running-statistics factor of this step (0.1 default; 1/num_batches_tracked when the
                            module's momentum is None) */
  const float* gamma;    /* [feat_dim] BatchNorm1d weight, NULL = 1 */
  const float* beta;     /* [feat_dim] BatchNorm1d bias, NULL = 0 */
  float* running_mean;   /* [feat_dim]; read in BN_EVAL, updated in BN_TRAIN (NULL = not tracked) */
  float* running_var;
  float* save_mean;      /* [feat_dim] statistics used by this call (BN modes): written by forward, read by backward */
  float* save_invstd;
  void* workspace;       /* BN modes: ffc_tail_workspace_bytes() bytes, 16-byte aligned, zero-filled once before its first use (calls
                            leave it reusable); one workspace must not be shared by calls that may run concurrently */
  int64_t workspace_bytes;
} ffc_tail_args;

int ffc_tail_workspace_bytes(int n_rows, int feat_dim, int64_t* bytes_out);
/* 1 launch (NORMALIZE) or 2 (BN modes). */
int ffc_tail_forward(const ffc_tail_args* a, void* stream);
/* Backward of ffc_tail_forward for the same `a` (x, p, inv_norm, save_* unchanged since forward): dp_dev rows dp_stride floats
 * apart; dx_dev [n_rows, feat_dim] contiguous.  dgamma_dev / dbeta_dev ([feat_dim], overwritten, either may be NULL) are the
 * BatchNorm1d weight / bias gradients (must be NULL in NORMALIZE mode).  1 launch (NORMALIZE) or 2. */
int ffc_tail_backward(const ffc_tail_args* a, const float* dp_dev, int64_t dp_stride, float* dx_dev, float* dgamma_dev,
                      float* dbeta_dev, void* stream);

/* fp32 -> bf16 mirror of n contiguous elements (queue initialisation / checkpoint load). */
int ffc_cast_bf16(const float* src_dev, void* dst_bf16_dev, int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused margin-softmax head pass (replaces ffc.py:195-202 / 248-254, add_margin ffc.py:60-138 and
 * its autograd backward): loss = add_margin(p . queue[0]^T, label) + add_margin(p . W2^T, label),
 * W2 = queue[1] on the `ones` slots and queue[0] elsewhere, plus dLoss/dp -- without materialising
 * the B x Q logits.  One sweep over the (local shard of the) queue accumulates, per probe row, the
 * softmax denominator, sum_j softmax_j * W_j (the embedding gradient) and the running top-k of the
 * hard-negative term; columns that differ between the two losses (`ones`) and each row's target
 * column are excluded from the sweep and handled in two small side sweeps / gather-dots.
 * ---------------------------------------------------------------------------------------------- */
typedef struct ffc_head ffc_head_t;

typedef struct ffc_head_config {
  int32_t max_rows;      /* max probe rows per pass (all ranks' rows when sharded) */
  int64_t q_local;       /* queue rows (slots) held by this rank */
  int64_t q_total;       /* global queue size (== q_local on one GPU) */
  int64_t col_offset;    /* global slot index of local row 0 */
  int32_t feat_dim;      /* D: 64, 128, 256 or 512 for the bf16 path; any multiple of 4 up to 512 in check mode */
  int32_t loss_type;     /* FFC_LOSS_* */
  float scale;           /* ffc.py:34 */
  float margin;          /* ffc.py:35 */
  int32_t topk;          /* ffc.py:48 hard_neg, 1..FFC_TOPK_MAX */
  int32_t precision;     /* FFC_PREC_* */
} ffc_head_config;

int ffc_head_create(const ffc_head_config* cfg, ffc_head_t** out);
int ffc_head_destroy(ffc_head_t* h);

/* Inputs of one pass; all device pointers. */
typedef struct ffc_head_pass {
  const float* p_f32;          /* [n_rows, D] probe embeddings (unit norm, ffc.py:157/209) */
  const float* queue_f32;      /* [2, q_local, D] */
  const void* queue_bf16;      /* [2, q_local, D] bf16 mirror (bf16 path) */
  const int32_t* label;        /* [n_rows] global slot or -1 (ffc.py:194/246) */
  const int32_t* ones_list;    /* [<= max_rows] LOCAL slots hit in this pass's bookkeeping (ffc.py:197) */
  const int32_t* n_ones;       /* device scalar */
  const uint32_t* cmask;       /* bitmask over LOCAL slots: bit set <=> slot in ones_list; may be NULL iff n_ones==0 always */
  int32_t n_rows;
} ffc_head_pass;

/* Rank-local statistics produced by the sweep, consumed by finalize.  Layout (all fp32 unless
 * noted), n = n_rows, k = topk, D = feat_dim:
 *   lsum   [4][n]      softmax denominators (relative to the fixed max M = c*scale): common under loss 1,
 *                      common under loss 2 (written and read only for SV), side0 (`ones` rows of queue[0]), side1 (queue[1])
 *   osum   [4][n][D]   sum_j p~_ij W_j for the same four column sets
 *   tgt    [4][n]      cos_t under queue[0], cos_t under W2, (owner flag as 1.0/0.0), spare
 *   topv   [3][n][k]   running top-k cosines (descending; -inf padded), topi int32 [3][n][k] GLOBAL slots
 * On several GPUs the caller sums lsum/tgt across ranks (all-reduce), all-gathers topv/topi, then
 * calls finalize, then reduce-scatters dp.  ffc_head_stats_bytes gives the sizes. */
typedef struct ffc_head_stats {
  float* lsum;
  float* osum;
  float* tgt;
  float* topv;
  int32_t* topi;
} ffc_head_stats;

int ffc_head_sweep(ffc_head_t* h, const ffc_head_pass* in, const ffc_head_stats* out, void* stream);

/* ffc_head_sweep in two steps, for the SV loss on a sharded queue (ffc.py:116-138): SV's hard-example threshold is the row's
 * target cosine minus the margin (ffc.py:121-122), and on R > 1 ranks only the owner of the target column can compute it.
 * ffc_head_prep writes out->tgt (target cosines, owner flag; zero where the target is not local); the caller sums tgt over the
 * ranks (all-reduce); ffc_head_sweep_prepared re-derives the thresholds from the summed tgt and runs the sweeps.  For AM / Arc
 * the pair is equivalent to ffc_head_sweep (the sweeps do not read tgt).  `in` / `out` must be the same in both calls. */
int ffc_head_prep(ffc_head_t* h, const ffc_head_pass* in, const ffc_head_stats* out, void* stream);
int ffc_head_sweep_prepared(ffc_head_t* h, const ffc_head_pass* in, const ffc_head_stats* out, void* stream);

/* Finalize: loss_out[0] = this pass's loss (both add_margin terms) -- identical on every rank when
 * stats were reduced; dp_out [n_rows, D] fp32 = this rank's contribution to dLoss/dp (the whole
 * gradient on one GPU).  n_ranks_topk: number of gathered top-k candidate sets in stats->topv/topi
 * ([n_ranks][3][n][k]); 1 on one GPU.  n_pos/n_out (global counts of label!=-1 / ==-1 rows) are
 * computed on the device from `label`. */
int ffc_head_finalize(ffc_head_t* h, const ffc_head_pass* in, const ffc_head_stats* stats,
                      int n_ranks_topk, float* loss_out, float* dp_out, void* stream);

/* One-GPU fast path: ffc_head_sweep + ffc_head_finalize(n_ranks_topk = 1) as one call.  On the bf16 AM / Arc path the chunk
 * reduction, the scalar part and dLoss/dp run as ONE kernel after the sweep (the statistics never round-trip through HBM, so
 * `scratch` is left partly unwritten: only tgt is filled); other configurations run the two calls back to back.
 * Replaces ffc.py:195-202 / 248-254 + loss.backward() of one head pass. */
int ffc_head_pass_single(ffc_head_t* h, const ffc_head_pass* in, const ffc_head_stats* scratch,
                         float* loss_out, float* dp_out, void* stream);

/* Sharded head (ffc_b200/dist.py; nothing like it in the reference): instead of ffc_head_sweep + all-reduce + all-gather +
 * ffc_head_finalize, a rank writes ONE record per pass (softmax denominators, target cosines, top-k candidates;
 * ffc_head_record_words 4-byte words), the records of all ranks are exchanged by one all-gather, and
 * ffc_head_finalize_gathered sums the scalars in rank order and produces this rank's partial dLoss/dp straight from its
 * sweep partials.  bf16 AM / Arc only. */
int ffc_head_record_words(const ffc_head_config* cfg, int n_rows, int64_t* words_out);
/* Record exchange by peer stores instead of an all-gather (ranks whose gathered-record buffers are peer-mapped, e.g. torch symmetric
 * memory): copies the record of the pass just swept (`record_dev`, as written by ffc_head_sweep_record on handle `h`) into every rank's
 * buffer at peer_ptrs_dev[r] + dst_offset_words -- the per-row scalars always, the top-k candidate slots only for rows whose label is -1
 * (the only rows whose candidates ffc_head_finalize_gathered reads; identical on every rank because the labels are).  Follow all pushes
 * of a step with ONE ffc_peer_barrier; the finalize calls after it may read the gathered buffer. */
int ffc_head_push_record(ffc_head_t* h, int n_rows, const float* record_dev, float* const* peer_ptrs_dev, int64_t dst_offset_words, int n_ranks,
                         void* stream);
int ffc_head_sweep_record(ffc_head_t* h, const ffc_head_pass* in, void* record_out, void* stream);
int ffc_head_finalize_gathered(ffc_head_t* h, const ffc_head_pass* in, const void* records, int n_ranks,
                               int64_t record_stride_words, float* loss_out, float* dp_out, void* stream);

/* ffc_head_finalize_gathered with the two extensions of the sharded head's merged step (ONE exchange point per FFC.forward):
 *   overlay_*: the finalize of a pass whose queue rows have been rewritten since its sweep (restore, the next pass's enqueue) reads
 *     those rows where their sweep-time content still is (see ffc_queue_scatter_overlay); NULL map = read the queue.
 *   dp_peer: device array of n_ranks pointers to the ranks' peer-mapped staging buffers.  Row i of this rank's partial dLoss/dp is
 *     stored to dp_peer[i / dp_rows_per_rank] + dp_slot_offset + (i % dp_rows_per_rank) * D -- straight into the owner rank's memory
 *     over NVLink, from the kernel that computes it -- instead of dp_out (which may then be NULL); after a barrier across the ranks
 *     the owner adds the n_ranks slabs with ffc_sum_slabs.  This is the reduce-scatter of dLoss/dp folded into finalize. */
typedef struct ffc_head_finalize_opts {
  const int32_t* overlay_map;
  const float* overlay_g;      /* table 0 rows: the gathered gallery embeddings of the pass, [.., D] fp32 */
  const float* overlay_undo;   /* table 1 rows: the undo buffer of the enqueue that followed, [.., D] fp32 */
  float* const* dp_peer;
  int32_t dp_rows_per_rank;
  int64_t dp_slot_offset;      /* in floats */
} ffc_head_finalize_opts;
int ffc_head_finalize_gathered_ex(ffc_head_t* h, const ffc_head_pass* in, const void* records, int n_ranks,
                                  int64_t record_stride_words, const ffc_head_finalize_opts* opts, float* loss_out,
                                  float* dp_out, void* stream);

/* Optional mode, off by default: dLoss/dQueue.  The reference keeps `queue` a no-grad buffer (ffc.py:29); a caller that trains the
 * prototypes enables the mode before a pass (ffc_head_set_dqueue: the fused finalize then also exports its per-row coefficients)
 * and, after the finalize of that pass (ffc_head_pass_single, ffc_head_finalize or ffc_head_finalize_gathered[_ex]) and before the
 * queue rows change again, calls ffc_head_dqueue: dqueue_out [2, q_local, D] fp32 is OVERWRITTEN with d(loss of the pass)/d(queue)
 * for an upstream gradient of 1 -- both add_margin terms (ffc.py:195-202 through autograd, had `queue` required grad) incl. the
 * hard-negative rows.  Every loss type (SV: the hard mask is not differentiated, its 1.2 z + 0.2 transform is) and both precisions.
 * bf16: one more sweep of the tcgen05 kernel with the roles of queue and probe rows swapped (4 n Q D FLOPs, no B x Q matrix) plus two
 * small kernels for the target / `ones` rows and the hard negatives; needs `in->queue_bf16`.  Check mode (FFC_PREC_FP32): SIMT
 * kernels with fp64 accumulation in a fixed order, bit-identical from run to run; needs `in->p_f32` and `in->queue_f32`.  On a shard
 * the result covers the handle's q_local slots: rows [col_offset, col_offset + q_local) of the gradient of the global queue, since
 * every rank sweeps all gathered probe rows and finalize's per-row coefficients are global.  `in` = the pass just finalized. */
int ffc_head_set_dqueue(ffc_head_t* h, int enable);
int ffc_head_dqueue(ffc_head_t* h, const ffc_head_pass* in, float* dqueue_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * 1:N identification against the resident prototypes (nothing like it in the reference: its test
 * chapter is empty).  The gallery of handle `h` is row queue[0][s] of every slot s < cur_idx of `lru`
 * (the LRU whose slots index this handle's queue; [0, cur_idx) is exactly the occupied set).  For each
 * query row: the k prototypes of highest cosine, ordered by score descending, ties by smaller slot.
 * score_out [n, k] fp32: fp64-accumulated dot of the query row with the fp32 queue row (x_f32 rows are
 * expected L2-normalised); label_out [n, k] int64: the slot's key; slot_out [n, k] int32: GLOBAL slot
 * (col_offset + local slot).  Fewer than k resident: the missing entries are slot -1, label INT64_MIN,
 * score -inf.  bf16 handles select the candidates by the tcgen05 bf16 cosine and rescore them; check-mode
 * handles (FFC_PREC_FP32) select by the fp32 score itself.  Reads the LRU's device state (cur_idx,
 * slot keys) without touching recency, and writes nothing but the outputs and the workspace.  No host sync;
 * two kernel launches per call (bf16: plus one memset), whatever n and cur_idx are.  1 <= k <= FFC_TOPK_MAX,
 * 1 <= n <= FFC_IDENTIFY_MAX_ROWS (callers split larger inputs).
 * ---------------------------------------------------------------------------------------------- */
#define FFC_IDENTIFY_MAX_ROWS 65536
int ffc_identify_workspace_bytes(ffc_head_t* h, int n, int k, int64_t* bytes_out);
/* x_f32: [n, D] unit rows.  Searches this handle's q_local slots [0, cur_idx of `lru`); slot_out holds GLOBAL slots.
 * queue_f32 / queue_bf16: [2, q_local, D] as for a head pass (queue_bf16 may be NULL in check mode); workspace: device memory of
 * ffc_identify_workspace_bytes bytes, 256-byte aligned, not shared with a call that may run concurrently. */
int ffc_identify(ffc_head_t* h, const ffc_lru_t* lru, const float* x_f32, int n, int k, const float* queue_f32,
                 const void* queue_bf16, void* workspace, int64_t workspace_bytes,
                 float* score_out, int64_t* label_out, int32_t* slot_out, void* stream);

/* sizes in bytes of the five stats arrays for n rows (one rank's worth) */
int ffc_head_stats_bytes(const ffc_head_config* cfg, int n_rows, int64_t sizes_out[5]);

/* Roofline evidence: when enabled, every MAIN sweep launch (the tcgen05 kernel over queue[0]) is
 * bracketed by CUDA events on its launch stream; get_timing (host-sync) returns the summed device
 * time in ms and the number of launches since set_timing(1). */
int ffc_head_set_timing(ffc_head_t* h, int enable);
int ffc_head_get_timing(ffc_head_t* h, double* total_ms_out, int64_t* launches_out);

/* Debug / evidence: number of kernel launches issued by this library since load. */
int64_t ffc_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* FFC_B200_H_ */
