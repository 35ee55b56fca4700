/* foodrec_b200.h -- C ABI of the B200-native Market2Dish Recommender hot path.
 *
 * The reference (WenjieWWJ/FoodRec, Code/Recommender) has no FFI/plugin layer:
 * its hot path is the TF-1.x graph built by Model_Recommender.py and driven by
 * sess.run() from Train_recommender.py / evaluate.py.  This header is the
 * boundary the Python `foodrec_b200.Model` / `Session` shim binds (ctypes); each
 * entry point cites the reference graph section it replaces.
 *
 * Conventions
 *  - plain pointers and sizes only; no torch/CUDA types (fr_stream == cudaStream_t
 *    passed as void*).
 *  - the caller owns every table and batch buffer (device memory unless the
 *    entry point says "host"); the library owns only its workspace.
 *  - every call is asynchronous and ordered on the given stream; returns FR_OK
 *    or a negative code and never throws; fr_last_error() gives the message.
 *  - one handle per device, not thread-safe; multi-GPU = one process per GPU.
 *  - no CPU fallback: a missing/failed CUDA device is an error.
 *
 * Layouts (all row-major, fp32 tables, int32 ids -- as in the reference):
 *   P   Personal_Memory   [U,5,D]  slot 0 = category memory, 1..4 = dish memories
 *   R   Recipe_Embedding  [I,D]
 *   Cat Category_Embedding[4,D]
 *   G   General_Memory    [L,5,D]
 * D must be a multiple of 4 and <= 256; all table pointers 16-byte aligned.
 */
#ifndef FOODREC_B200_H
#define FOODREC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FR_ABI_VERSION 1

typedef struct fr_ctx* fr_handle;
typedef void* fr_stream; /* cudaStream_t */

enum { FR_OK = 0, FR_ERR_ARG = -1, FR_ERR_CUDA = -2, FR_ERR_STATE = -3, FR_ERR_UNSUPPORTED = -4 };

/* Model_Recommender.py:228-235 -- learner is matched case-insensitively, anything else = SGD */
enum { FR_SGD = 0, FR_ADAGRAD = 1, FR_RMSPROP = 2, FR_ADAM = 3 };
/* TF-1.x sparse Adam decays m,v and moves var for EVERY row each step (adam.py
 * _apply_sparse_shared).  DENSE does that sweep literally; LAZY_EXACT defers it per
 * row (last-step stamp) and replays the skipped steps with identical arithmetic
 * when the row is next touched or on fr_adam_flush -- same results, O(touched) traffic.
 * LAZY_SERIES replaces the step-by-step replay of the k skipped steps by their closed form
 *   sum_j lr_j b1^j m / (sqrt(b2^j v) + eps) = m/(q+eps) * sum_n C_n y^n ,  y = q/(q+eps), q = sqrt(v),
 *   C_n = sum_j lr_j b1^j (1 - b2^(j/2))^n   (row-independent; kept per last-step in a table)
 * truncated at n = 4: relative error of the catch-up term < 1e-9 for any k (the b1^j weights
 * kill the slowly converging late terms), i.e. below fp32 round-off -- O(1) work per element
 * instead of O(k).  Results equal DENSE to fp32 rounding (tests: 1e-5 parity bound). */
enum { FR_ADAM_DENSE = 0, FR_ADAM_LAZY_EXACT = 1, FR_ADAM_LAZY_SERIES = 2 };
enum { FR_POINTWISE = 0, FR_BPR = 1 };

/* Mirrors the args fields Model.__init__ reads (Model_Recommender.py:6-24). */
typedef struct {
  int32_t embed_size;   /* D */
  int32_t num_users;    /* U (rows of P held by this process) */
  int32_t num_items;    /* I (rows of R held by this process) */
  int32_t num_labels;   /* L */
  int32_t learner;      /* FR_SGD.. */
  int32_t adam_mode;    /* FR_ADAM_* */
  int32_t max_rows;     /* capacity: item rows per step (B pointwise, 2B BPR) */
  int32_t max_label_entries; /* capacity: non-zeros of the label feed per step */
  float lr;                             /* args.lr (global_step never advances: lr is constant, :224-226) */
  float high_level_score_coefficient;   /* a, :17 ; low coefficient = 1-a, :96 */
  float beta_1, beta_2, alpha;          /* write coefficients :115,:140,:196 */
  float clip_norm;                      /* 5.0, :237 */
  float adam_beta1, adam_beta2, adam_eps;
  float rms_decay, rms_eps;
} fr_config;

/* Device tables + optimizer slots (caller-owned).  Slot meaning by learner:
 *   ADAM: s1=m (0), s2=v (0);  ADAGRAD: s1=accumulator (0.1);  RMSPROP: s1=ms (1), s2=mom (0)
 * last_* (int32 per row, 0-initialised) are required for FR_ADAM only. */
typedef struct {
  float *P, *R, *Cat, *G;
  float *s1_P, *s2_P, *s1_R, *s2_R, *s1_Cat, *s2_Cat;
  int32_t *last_P, *last_R;
  /* optional device-resident side tables for the compact (ids-only) feed:
   * item_cats [I,4] = dish_to_category; label CSR over users = user_to_one_hot_label */
  const float* item_cats;
  const int32_t* user_label_off; /* [U+1] */
  const int32_t* user_label_idx; /* [nnz], values in [0,L) , weight 1 */
} fr_tables;

/* One batch = the placeholders of Model_Recommender.py:26-33.
 * n_groups = B.  Item rows: pointwise S=B (row b); BPR S=2B (row 2t = positive,
 * 2t+1 = negative of triple t).  NULL selects the compact alternative. */
typedef struct {
  int32_t mode;            /* FR_POINTWISE | FR_BPR */
  int32_t n_groups;        /* B */
  const int32_t* users;    /* [B]    user_input */
  const int32_t* items;    /* [S]    item_input (BPR: interleaved pos/neg) */
  const float* cats;       /* [S,4]  categories ([.,4,1] flattened); NULL -> tables.item_cats[item] */
  const float* labels;     /* [B]    labels (pointwise only) */
  const float* write_sign; /* [S]    write_sign; NULL -> +1 if label>0.5 else -1 (BPR: +1 pos, -1 neg) */
  const float* user_labels;/* [B,L]  user_one_hot_label; NULL -> tables.user_label_* CSR by user */
} fr_batch;

/* Device scalars written by fr_train_step (index into float out[FR_OUT_COUNT]). */
enum { FR_OUT_LOSS = 0, FR_OUT_NORM = 1, FR_OUT_SCALE = 2, FR_OUT_GENERAL = 3,
       FR_OUT_PERSONAL = 4, FR_OUT_LR = 5, FR_OUT_UNIQ_USERS = 6, FR_OUT_UNIQ_ITEMS = 7,
       FR_OUT_LABEL_ENTRIES = 8,
       FR_OUT_OVERFLOW = 9 /* 1: label feed exceeded max_label_entries; 2: fr_shard.cap exceeded; 3: a user / recipe id
                              outside its table (the row was redirected to row 0: the step's results are invalid) */,
       FR_OUT_COUNT = 12 };

int fr_abi_version(void);
int fr_create(const fr_config* cfg, fr_handle* out);
int fr_destroy(fr_handle h);
const char* fr_last_error(fr_handle h);
int fr_set_tables(fr_handle h, const fr_tables* t);

/* Storage format of Personal_Memory and Recipe_Embedding (BASELINE configs[4]: bf16 tables).  FR_TABLE_BF16: tables.P and
 * tables.R point to bf16 rows (same shapes, 2 bytes per element, 8-byte aligned); Category_Embedding, General_Memory and
 * the optimizer slots stay fp32.  All arithmetic is fp32: a row is converted on load and ROUNDED TO NEAREST EVEN ON STORE
 * (the rule oracle/recommender_oracle.py states and the CUDA path is tested against).  Offered for the natively sparse
 * optimizers (SGD, Adagrad, RMSProp): TF-1.x Adam moves EVERY row EVERY step, which has no sensible meaning on rows that
 * are re-rounded to 8 bits of mantissa each time (updates below half an ulp vanish) -- FR_ADAM returns FR_ERR_UNSUPPORTED.
 * Not available with bf16 tables: personal-write steps, fr_catalog_* (its exact re-rank reads fp32 rows), fr_set_shadow.
 * The row-sharded phases exchange recipe rows in fp32 (the owner's gather converts).  Call before fr_set_tables. */
enum { FR_TABLE_F32 = 0, FR_TABLE_BF16 = 1 };
int fr_set_table_format(fr_handle h, int32_t format);

/* Single-pass training step (lazy Adam only).  The two-pass step reads Personal_Memory and its Adam slots twice per
 * step -- once to score, once to update -- because tf.clip_by_global_norm (Model_Recommender.py:237) separates the
 * gradient from apply_gradients.  With a second, caller-owned copy of P / m / v ([U,5,D] each, contents irrelevant)
 * fr_train_step scores AND updates a user's rows in one kernel, speculating that the clip is inactive (scale == 1):
 * new rows go to the other copy and become current (one bit of the row's last_P stamp) only once the norm is known;
 * if the clip is active the step falls back to the two-pass update with the true scale -- results are those of the
 * two-pass step either way.  While enabled, the caller's P / s1_P / s2_P may be stale for some rows between calls:
 * every library entry point that reads them brings them up to date first, and fr_adam_flush does so for the caller.
 * Passing three NULLs switches it off again.  Not used by the row-sharded phases (fr_shard_*). */
int fr_set_shadow(fr_handle h, float* P_alt, float* s1_P_alt, float* s2_P_alt);

/* Optimizer step counter (TF: the beta-power accumulators of adam.py); set on restore. */
int fr_get_step(fr_handle h, int64_t* step);
int fr_set_step(fr_handle h, int64_t step);

/* Health term at inference (BASELINE configs[4]): when enabled, fr_fwd_score, fr_eval_sampled_topk and
 * fr_catalog_topk score every user with  P'[u] = P[u] + alpha * mean_{l in labels(u)} G[l]  -- the row
 * Write_Memory materialises on a personal step (Model_Recommender.py:170-198) -- gathered and blended inside
 * the kernels, nothing is written.  Needs tables.user_label_off/idx.  Training is unaffected. */
int fr_set_health_blend(fr_handle h, int32_t enable);

/* inference, Model_Recommender.py:56-97 -> scores[n].  cats NULL -> item_cats table. */
int fr_fwd_score(fr_handle h, const int32_t* users, const int32_t* items, const float* cats,
                 int32_t n, float* scores, fr_stream s);

/* One sess.run([loss_value, learning_rate, (personal,) general, train_op]) --
 * Train_recommender.py:182-199: inference :56-97, loss :99-104, compute_gradients +
 * clip_by_global_norm + apply_gradients :223-241, Write_Memory :106-220
 * (write_personal != 0 <=> the run fetches model.personal).
 * out_scalars: device float[FR_OUT_COUNT]; out_scores: device float[S] or NULL. */
int fr_train_step(fr_handle h, const fr_batch* b, int32_t write_personal,
                  float* out_scalars, float* out_scores, fr_stream s);

/* Same step with HOST batch buffers and a HOST out_scalars[FR_OUT_COUNT] (pinned for
 * true async): H2D of the feed and D2H of the scalars are issued on the stream. */
int fr_train_step_host(fr_handle h, const fr_batch* host_batch, int32_t write_personal,
                       float* host_out_scalars, fr_stream s);

/* Input prefetch for the host-buffer path: starts the host->device copy of a FUTURE batch on the library's
 * own copy stream (two staging slots) and returns at once; the next fr_train_step_host call that is given the
 * same fr_batch (same host pointers, mode and size) skips its own copies and only waits for that one.  Lets the
 * PCIe transfer of batch k+1 overlap the kernels of batch k.  The host buffers must stay untouched (and should
 * be pinned) until that step has been queued. */
int fr_feed_prefetch(fr_handle h, const fr_batch* host_batch);

/* Per-phase device time of fr_train_step, measured with CUDA events recorded on the
 * step's stream (the measurement bench.py's roofline uses).  fr_timing_read waits for
 * the outstanding events and returns, per phase, the summed milliseconds over n_steps.
 * fr_shard_update records the same set for its own kernels (user pass and its combine, local recipe-gradient pass;
 * FR_T_LABEL there = personal pass + dG add); phases that live in other fr_shard_* calls read as zero. */
enum { FR_T_SORT = 0, FR_T_FWD = 1, FR_T_FINALIZE = 2, FR_T_USER_CHUNK = 3, FR_T_USER_COMBINE = 4,
       FR_T_LABEL = 5, FR_T_ITEM_CHUNK = 6, FR_T_ITEM_COMBINE = 7, FR_T_SWEEP = 8, FR_T_MISC = 9,
       FR_T_COUNT = 10 };
/* number of CUDA kernels this library has launched in this process (bench.py gpu_launches) */
int64_t fr_launch_count(void);
int fr_timing_enable(fr_handle h, int32_t enable);
int fr_timing_read(fr_handle h, double* ms_sum /* [FR_T_COUNT] */, int64_t* n_steps, int32_t reset);

/* Bring every row of P and R to the current step (LAZY_EXACT); no-op otherwise.
 * Must precede any read of the tables by the caller (eval, checkpoint). */
int fr_adam_flush(fr_handle h, fr_stream s);

/* evaluate.py:35-66 batched: per test user, candidates cand[u, 0..n_cand[u]) (first =
 * held-out positive), dict-dedup + heapq.nlargest(K) semantics (ties keep insertion
 * order).  Outputs: topk_ids [n_users,K] (-1 padded), gt_rank [n_users] (position of the
 * positive in the ranklist or -1), scores [n_users,cand_stride] or NULL. */
int fr_eval_sampled_topk(fr_handle h, const int32_t* users, const int32_t* cand,
                         const int32_t* n_cand, int32_t n_users, int32_t cand_stride,
                         const float* cand_cats /* [n_users,cand_stride,4] or NULL */,
                         int32_t K, int32_t* topk_ids, int32_t* gt_rank, float* scores,
                         fr_stream s);

/* ---- Row-sharded training: one process per GPU (torchrun), W <= 8 ranks.
 * Personal_Memory (+slots) is sharded by user % W -- samples are routed to the user owner
 * when they are loaded, so the 5D-float user rows and their updates never move;
 * Recipe_Embedding (+slots) is sharded by recipe % W; Category_Embedding and General_Memory
 * are replicated.  fr_config.num_users / num_items are the LOCAL row counts.
 * batch.users are LOCAL user rows (user / W), batch.items GLOBAL recipe ids.
 * One step = five phases separated by the caller's collectives (torch.distributed / NCCL):
 *
 *   fr_shard_plan     sort rows, dedup recipes per owner -> req[W*cap] (row at owner, -1 empty)
 *     all_to_all(req)                                     -> rreq
 *   fr_shard_serve    owner: catch up (lazy Adam) and gather the requested rows -> rows[W*cap,D]
 *     all_to_all(rows)                                    -> rbuf
 *   fr_shard_forward  forward/loss/norm partials + General_Memory delta -> packed[fr_shard_packed_len]
 *     all_reduce(packed, SUM)        {loss, sum|g|^2, dCat[4,D], dG[L,5,D]}
 *   fr_shard_update   clip scale, Cat, Personal_Memory pass, G += dG, recipe gradient rows -> grows[W*cap,D]
 *     all_to_all(grows)                                   -> rgrows
 *   fr_shard_apply    owner: segment-reduce the received gradient rows by recipe + optimizer
 *
 * cap = per-(source,owner) capacity in unique recipes; overflow sets FR_OUT_OVERFLOW = 2.
 * All buffers are device memory owned by the caller. */
typedef struct {
  int32_t world, rank, cap;
  int32_t items_per_rank;   /* ceil(I / world): local rows of Recipe_Embedding */
  int32_t global_batch;     /* groups summed over ranks: the loss mean divides by it */
} fr_shard;
int64_t fr_shard_packed_len(fr_handle h);
/* Routing of a batch that was NOT loaded at its users' owners (batch.users = GLOBAL user ids): every group is written,
 * in batch order, into the block of the rank that owns its user (user % world): send [world][block], block =
 * fr_shard_route_block(batch, rcap) int32 = [rcap local user rows | rcap*group recipe ids | (pointwise) rcap labels as
 * bits], -1 padded.  The caller exchanges the blocks with ONE all-to-all; fr_shard_unroute compacts what arrived, in
 * (source rank, position) order, into a routed batch (users = local rows) and writes its size to n_out (device int32:
 * the caller reads it to call fr_shard_plan).  More than rcap groups for one destination, or more than cap_out
 * received, raise *out_flag = 2 (NULL: the step's FR_OUT_OVERFLOW). */
int64_t fr_shard_route_block(const fr_batch* b, int32_t rcap);
int fr_shard_route(fr_handle h, const fr_batch* b, int32_t world, int32_t rcap, int32_t* send, float* out_flag, fr_stream s);
int fr_shard_unroute(fr_handle h, int32_t mode, int32_t world, int32_t rcap, const int32_t* recv, int32_t cap_out,
                     int32_t* users, int32_t* items, float* labels, int32_t* n_out, float* out_flag, fr_stream s);
/* Optional, one step ahead: the owner-side ordering of the request list fr_shard_serve / fr_shard_apply walk (keys +
 * stable sort by recipe) depends on the requests only, not on the tables, so it may be issued -- on another stream --
 * right after the id all-to-all of the step fr_shard_plan planned last, while the previous step is still running
 * (two sets of buffers, like the plan slots).  fr_shard_serve does it itself when this was not called. */
int fr_shard_serve_prepare(fr_handle h, const fr_shard* sh, const int32_t* rreq, fr_stream s);

/* Peer-memory exchange over NVLink instead of the two row all-to-alls: peer_rbuf[w] / peer_rgrows[w] are rank w's
 * receive buffers ([W*cap, D] each) mapped into this process (CUDA IPC; the caller's own buffers at index rank).
 * Afterwards fr_shard_serve(rows = NULL) stores every gathered recipe row straight into the requester's rbuf and
 * fr_shard_update(grows = NULL) every finished gradient row into its owner's rgrows -- the place the all-to-all
 * would have put it.  The caller replaces each all-to-all by a barrier (all ranks have finished the phase). */
int fr_shard_set_peers(fr_handle h, const fr_shard* sh, float* const* peer_rbuf, float* const* peer_rgrows);
int fr_shard_plan(fr_handle h, const fr_batch* b, const fr_shard* sh, int32_t* req, fr_stream s);
int fr_shard_serve(fr_handle h, const fr_shard* sh, const int32_t* rreq, float* rows, fr_stream s);
int fr_shard_forward(fr_handle h, const fr_batch* b, const fr_shard* sh, const float* rbuf, float* packed,
                     fr_stream s);
int fr_shard_update(fr_handle h, const fr_batch* b, const fr_shard* sh, int32_t write_personal, const float* rbuf,
                    const float* packed_reduced, float* grows, float* out_scalars, fr_stream s);
int fr_shard_apply(fr_handle h, const fr_shard* sh, const int32_t* rreq, const float* rgrows, float* out_scalars,
                   fr_stream s);

/* ---- Full-catalog top-K (extension; definition = inference :56-97 over EVERY recipe, the
 * K best by (score desc, id asc)).  The dense contraction runs in bf16 on tcgen05 as a FILTER
 * with a proven error bound; survivors are re-scored in fp64 from the fp32 tables, so ids are
 * exact and scores are the fp64 value of the reference formula (see csrc/catalog.cuh).
 * Requires tables.item_cats with 0/1 entries (dish_to_category); recipes with no category are
 * never returned (the reference divides by zero for them, Model_Recommender.py:79,92).
 *
 * fr_catalog_prepare builds the recipe-side index from the CURRENT R / item_cats (recipes
 * grouped by category mask, bf16 operand, norms).  It synchronises the stream and must be
 * called again after R or item_cats change.  P and Cat are read at query time. */
typedef struct {
  int32_t cta_group;      /* 0 = default (2: CTA pairs, tcgen05 cta_group::2), 1 = single-CTA MMA */
  int32_t max_pass_rows;  /* 0 = default; users processed per pass */
  int32_t splits;         /* 0 = auto; pieces the recipe sweep is cut into for small user counts */
  int32_t epi_sets;       /* 0 = default (1); 1, 2 or 4 epilogue warp sets (each owns tile_n/sets accumulator columns
                             and keeps its own candidate list per user) */
  int32_t tile_n;         /* 0 = default (256: 2 accumulator stages in TMEM); 128: 4 stages */
  int32_t a_split;        /* 0 = default: user operand as bf16 head + tail (two MMAs per recipe block, halves the
                             filter's error bound) when D <= 128; 1 = single bf16 operand */
} fr_catalog_opts;
int fr_catalog_prepare(fr_handle h, const fr_catalog_opts* opts, const float* item_cats /* [num_items,4] of THIS
                       table's rows, or NULL = tables.item_cats (a row-sharded table passes its local slice) */,
                       fr_stream s);
/* Query rows: P_rows != NULL -> dense device rows [n_users,5,D] (e.g. all-gathered from the user
 * owners); else users[n_users] (device) index tables.P, NULL = 0..n_users-1.
 * out_ids [n_users,K] = local recipe row * id_mul + id_add (-1 padded); out_scores [n_users,K]
 * fp64 or NULL.  Asynchronous on the stream. */
int fr_catalog_topk(fr_handle h, const int32_t* users, const float* P_rows, int32_t n_users, int32_t K,
                    int32_t id_mul, int32_t id_add, int32_t* out_ids, double* out_scores, fr_stream s);
/* fr_catalog_topk that leaves out, per query row, the recipes the caller lists (e.g. the user's training positives):
 * the K best by (score desc, id asc) among the recipes that have a category and are NOT on the row's list, -1 / -inf
 * padded when fewer remain.  Lists are a CSR over query rows on the device: excl_off [n_users+1], excl_ids [nnz]
 * (int32; both NULL = no lists = fr_catalog_topk, bit for bit).  Ids are in the OUTPUT id space (local row * id_mul
 * + id_add), so a recipe shard takes the global lists unchanged; any order, duplicates allowed; an id this table
 * cannot return (another shard's, out of range, negative) is ignored.  The filter is widened per row by the row's
 * listed recipes of this table (csrc/catalog.cuh); a row with K + that count > 256 takes the exact fallback
 * (counted by fr_catalog_fallback_rows).  id_mul >= 1 with lists.  Asynchronous on the stream. */
int fr_catalog_topk_excluding(fr_handle h, const int32_t* users, const float* P_rows, int32_t n_users, int32_t K,
                              const int32_t* excl_off, const int32_t* excl_ids, int32_t id_mul, int32_t id_add,
                              int32_t* out_ids, double* out_scores, fr_stream s);
/* Dense copies of Personal_Memory rows: out[k] = P[users[k]] ([n,5,D], device) -- the query rows a rank contributes to
 * the all-gather of the item-sharded top-K (a user id outside the table yields a zero row). */
int fr_gather_user_rows(fr_handle h, const int32_t* users, int32_t n, float* out, fr_stream s);
/* Item-sharded merge: ids/scores [n_lists, n_users, K] (each list sorted, -1 padded) ->
 * the K best of the union by (score desc, id asc).  n_lists*K <= 4096. */
int fr_catalog_merge(fr_handle h, const int32_t* ids, const double* scores, int32_t n_lists, int32_t n_users,
                     int32_t K, int32_t* out_ids, double* out_scores, fr_stream s);
/* Device time per phase {user operand, tcgen05 GEMM+filter, exact re-rank, exact fallback},
 * CUDA events on the call's stream, recorded while fr_timing_enable is on. */
int fr_catalog_timing_read(fr_handle h, double* ms_sum /* [4] */, int64_t* n_passes, int32_t reset);
/* {cta_group, padded K, tiles, present-mask bits, recipes with a category, epilogue sets, list capacity, fallback blocks} */
int fr_catalog_info(fr_handle h, int32_t* out /* [8] */);
/* in-kernel cycle counters of the GEMM kernel (collected while the environment variable
 * FOODREC_CATALOG_CYCLES is set): {MMA thread total, waiting for a free accumulator, waiting for
 * operands, #MMA threads, epilogue warp total, waiting for an accumulator, #epilogue warps, 0}; resets. */
int fr_catalog_cycle_counters(fr_handle h, uint64_t* out /* [8] */, fr_stream s);
/* rows of the LAST pass that took the exact full-scan fallback (synchronises the stream) */
int fr_catalog_fallback_rows(fr_handle h, int32_t* out, fr_stream s);

/* ---- Negative sampling for 1:N BPR (extension; the reference only takes listed negatives,
 * Train_recommender.py:86-93).  Counter-based so host and device agree bit for bit:
 * Philox4x32-10 with counter (sample_lo, sample_hi, j, attempt), key = seed; item = mulhi32(x0, I);
 * a draw equal to the positive is re-drawn (<= 16 attempts, then (positive+1) % I).
 * pos_items [n] device; out [n, n_neg] device; sample index = sample_offset + row. */
int fr_sample_negatives(fr_handle h, const int32_t* pos_items, int64_t n, int32_t n_neg, uint64_t seed,
                        uint64_t sample_offset, int32_t* out, fr_stream s);
/* The same draws written as the expanded BPR batch fr_train_step / fr_shard_plan consume: for sample s and negative j,
 * triple t = s*n_neg + j gets out_users[t] = users[s], out_items[2t] = pos_items[s], out_items[2t+1] = the negative.
 * num_items = the size of the catalog the negatives are drawn from (0: this handle's Recipe_Embedding; a row-sharded
 * rank passes the GLOBAL recipe count).  out_users [n*n_neg], out_items [2*n*n_neg] (8-byte aligned), device. */
int fr_sample_bpr_batch(fr_handle h, const int32_t* users, const int32_t* pos_items, int64_t n, int32_t n_neg,
                        uint64_t seed, uint64_t sample_offset, int64_t num_items, int32_t* out_users,
                        int32_t* out_items, fr_stream s);
/* The raw generator (known-answer tests): ctr_key [n,6] = counter[4], key[2] -> out [n,4]. */
int fr_philox4x32_10(fr_handle h, const uint32_t* ctr_key, int32_t n, uint32_t* out, fr_stream s);

/* stable LSD radix sort of (key, index) pairs -- exported for tests of the
 * sort-and-segment machinery.  keys [n] (values < 2^nbits), out_keys/out_idx [n]. */
int fr_sort_pairs(fr_handle h, const uint32_t* keys, int32_t n, int32_t nbits,
                  uint32_t* out_keys, uint32_t* out_idx, fr_stream s);

#ifdef __cplusplus
}
#endif
#endif /* FOODREC_B200_H */
