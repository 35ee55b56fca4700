// Context of one fr_handle + small host helpers shared by api.cu and api_shard.cu.
#pragma once
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "train.cuh"

using namespace fr;
namespace fr { struct CatalogWs; }

struct fr_ctx {
  fr_config cfg{};
  fr_tables tab{};
  bool has_tables = false;
  ModelConsts mc{};
  int NV = 1, sm_count = 148, device = 0;
  size_t l2_persist_max = 0, l2_window_max = 0;   // device limits for a persisting-L2 access window (0: unsupported)
  bool l2_lines_pinned = false;                   // a kernel ran with a persisting window since the last reset
  int64_t step = 0;
  float b1p = 0.f, b2p = 0.f;
  char err[512] = {0};
  std::vector<void*> allocs;

  // workspace (device)
  uint32_t* ukeys = nullptr; int32_t *users_s = nullptr, *items_s = nullptr;   // range-checked copies of the step's ids
  float* ws_row = nullptr; float* g = nullptr; float* scores = nullptr;
  float4* z = nullptr;
  SortBufs sortU, sortI, sortL;
  float *part_loss = nullptr, *part_nrm = nullptr; float4* part_gcat = nullptr; int fwd_grid_cap = 0;
  float* packed = nullptr;
  float4 *pieces_u = nullptr, *pieces_i = nullptr, *pieces_g = nullptr, *pieces_personal = nullptr;
  size_t pieces_personal_chunks = 0;
  uint32_t *counts = nullptr, *offs = nullptr, *ent_key = nullptr, *ent_row = nullptr, *n_entries = nullptr;
  float* ent_coef = nullptr;
  uint32_t* counters = nullptr;        // [0] unique users, [1] unique recipes, [2]/[3] long chains (label / recipe pass)
  uint4* long_list = nullptr; uint32_t long_cap = 0;   // work list of seg_combine_long_kernel (train.cuh)
  float4* cat_pre = nullptr;
  float* lr_hist = nullptr; int64_t lr_hist_cap = 0;
  double* cser = nullptr;          // LAZY_SERIES coefficient table [lr_hist_cap * SERIES_TERMS]
  double* mean_partials = nullptr;
  float* out_internal = nullptr;
  uint32_t* scan_tmp = nullptr;
  // row-sharded training (api_shard.cu): allocated on first use
  // Per-step plan state of the row-sharded step.  TWO slots: fr_shard_plan of step k+1 may be issued (on another
  // stream) while forward / update / apply of step k are still running -- plan depends only on the batch ids, and with
  // the id all-to-all it is ~0.3 ms of small latency-bound kernels that hide under the previous step's update.
  // Slot 0 aliases the single-GPU step's buffers (ukeys, users_s, items_s, ws_row, sortU, sortI, out_internal).
  struct PlanSlot {
    size_t s_cap = 0;
    uint32_t* ukeys = nullptr; int32_t *users_s = nullptr, *items_s = nullptr; float* ws_row = nullptr;
    SortBufs sortU, sortI;
    uint32_t *okeys = nullptr, *flags = nullptr, *excl = nullptr, *owner_counts = nullptr, *slot_sorted = nullptr, *scan_tmp = nullptr;
    int32_t* slot_of_row = nullptr;
    float4* cats_row = nullptr;
    float* flag_out = nullptr;             // [FR_OUT_COUNT]: flags raised while planning / in forward, copied to `out` in update
    int ru = 0, ri = 0;                    // which sort buffer holds each result
    int mode = 0, B = 0, S = 0, group = 1;
    bool fused = false;                    // the step ran the single-pass forward (fr_shard_forward)
    bool planned = false;                  // fr_shard_plan has run for this slot's step (S may be 0: a rank that owns no row of the batch)
  };
  struct ShardWs {
    PlanSlot ps[2];
    uint64_t n_plan = 0, n_apply = 0;      // plan k writes slot k & 1; forward / update / apply of step k read slot k & 1
    size_t n_cap = 0;                      // W*cap the owner-side buffers are sized for
    uint32_t* route_counts = nullptr;
    // owner side: the received requests of a step sorted by recipe (keys, stable sort, count of valid slots).  Two
    // sets, like the plan slots: fr_shard_serve_prepare of step k+1 may run (side stream) while fr_shard_apply of
    // step k still reads step k's order.
    struct ServeSlot {
      uint32_t *serve_keys = nullptr, *n_valid = nullptr;
      SortBufs sortS;
      int rs = 0;
      bool prepared = false;
    } ss[2];
    float4* pieces_s = nullptr;
    fr::PeerPtrs peer_rbuf{}, peer_rgrows{};   // fr_shard_set_peers: NVLink P2P exchange instead of all-to-alls
  } sh;
  // sampled evaluation on row-sharded tables (eval_shard.cu): workspace of fr_shard_eval_plan for n_cap candidate
  // entries, re-allocated (after a stream synchronise) when a call needs more
  struct EvalPlanWs {
    size_t n_cap = 0;
    uint32_t *keys = nullptr, *flags = nullptr, *excl = nullptr, *scan_tmp = nullptr, *owner_counts = nullptr;
    SortBufs sort;
  } ev;
  // single-pass training (fr_set_shadow): second copy of Personal_Memory + Adam slots; shadow_dirty = some row's current
  // copy may be the shadow (cleared by shadow_sync, which every reader of the caller's tables runs first)
  float *shP = nullptr, *shM = nullptr, *shV = nullptr; bool shadow_dirty = false;
  bool table_bf16 = false;          // fr_set_table_format: Personal_Memory and Recipe_Embedding are stored in bf16
  bool health_blend = false;        // fr_set_health_blend: inference scores P[u] + alpha * mean G[labels(u)]
  fr::CatalogWs* cat = nullptr;     // full-catalog top-K (catalog.cu): index + pass workspace
  // fr_set_user_history: caller-owned CSR over Personal_Memory rows the sampler rejects negatives from (sampler.cu)
  const int32_t *hist_off = nullptr, *hist_ids = nullptr;
  uint32_t* hist_flag = nullptr;    // its validation flag
  // staging for fr_train_step_host
  void* stage = nullptr; size_t stage_bytes = 0;
  // fr_feed_prefetch: two staging slots filled on a private copy stream while the previous step computes
  struct FeedSlot {
    void* buf = nullptr; size_t bytes = 0;
    fr_batch host{}, dev{};            // identity of the staged host batch / its device image
    float* dout = nullptr;
    bool valid = false, used = false;
    cudaEvent_t copied = nullptr, consumed = nullptr;
  } feed[2];
  cudaStream_t copy_stream = nullptr;
  // fork / join inside fr_train_step: the label feed's entry list (count, scan, emit, sort by label) depends only on the
  // batch and is built on this stream while the sorts, catch-up and the forward run on the caller's
  cudaStream_t aux_stream = nullptr; cudaEvent_t aux_fork = nullptr, aux_fork2 = nullptr, aux_join = nullptr;
  cudaStream_t aux2_stream = nullptr; cudaEvent_t aux2_fork = nullptr, aux2_join = nullptr;      // finalize beside the fused kernel's combine
  int feed_next = 0;
  // per-phase timing (fr_timing_*)
  bool timing = false;
  struct TimingSet { cudaEvent_t ev[FR_T_COUNT + 1]; bool used = false; };
  std::vector<TimingSet> tsets;
  size_t ts_next = 0;
  double t_sum[FR_T_COUNT] = {0};
  int64_t t_steps = 0;
};

static inline void timing_collect(fr_ctx* h, fr_ctx::TimingSet& ts) {
  if (!ts.used) return;
  cudaEventSynchronize(ts.ev[FR_T_COUNT]);
  for (int i = 0; i < FR_T_COUNT; ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ts.ev[i], ts.ev[i + 1]) == cudaSuccess) h->t_sum[i] += ms;
  }
  h->t_steps += 1;
  ts.used = false;
}

// The phase events of one step on stream st (fr_timing_*); every call is a no-op while timing is off
struct StepTiming {
  fr_ctx::TimingSet* ts = nullptr;
  cudaStream_t st;
  StepTiming(fr_ctx* h, cudaStream_t s) : st(s) {
    if (!h->timing) return;
    ts = &h->tsets[h->ts_next++ % h->tsets.size()];
    timing_collect(h, *ts);
    ts->used = true;
  }
  void mark(int i) const { if (ts) cudaEventRecord(ts->ev[i], st); }
  cudaEvent_t ev(int i) const { return ts ? ts->ev[i] : nullptr; }
};

// Where the rows of a training step come from: the single-GPU step reads the tables, the row-sharded phases the rows
// this rank planned and received.  The phase builders below take everything else from the context.
struct StepRows {
  int B, S, group;
  const int32_t *users, *items;       // range-checked user rows; each row's recipe row in R
  const float* ws_row;                // write sign of each row
  const uint32_t *ukeys, *uperm;      // the rows sorted by user: keys, permutation
  const float4* R; bool R_is_table;   // the recipe rows read: Recipe_Embedding, or the received rows (always fp32)
  const float4* cats; int cats_by_item;
  const float *labels, *user_labels;  // the batch's
  float Bnorm;                        // divisor of the loss mean: the (global) batch size
  float* out;                         // flags and scalars
  float* scores;
  float4* G;                          // target of the label pass: General_Memory, or this rank's delta of it
};

static inline int fail(fr_ctx* h, int code, const char* fmt, ...) {
  if (h) {
    va_list ap; va_start(ap, fmt);
    vsnprintf(h->err, sizeof(h->err), fmt, ap);
    va_end(ap);
  }
  return code;
}
#define FR_CUDA(h, call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) \
  return fail(h, FR_ERR_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); } while (0)
#define FR_CHECK_LAUNCH(h) do { cudaError_t e_ = cudaGetLastError(); if (e_ != cudaSuccess) \
  return fail(h, FR_ERR_CUDA, "%s:%d kernel launch: %s", __FILE__, __LINE__, cudaGetErrorString(e_)); } while (0)

template <class T>
static inline int dalloc(fr_ctx* h, T** p, size_t count) {
  void* q = nullptr;
  if (count == 0) count = 1;
  cudaError_t e = cudaMalloc(&q, count * sizeof(T));
  if (e != cudaSuccess) return fail(h, FR_ERR_CUDA, "cudaMalloc(%zu bytes): %s", count * sizeof(T), cudaGetErrorString(e));
  h->allocs.push_back(q);
  *p = static_cast<T*>(q);
  return FR_OK;
}

// the step's side stream (highest priority: its CTAs are placed first when both streams have work) + fork/join events
static inline int aux_ensure(fr_ctx* h) {
  if (h->aux_stream) return FR_OK;
  int lo = 0, hi = 0;
  FR_CUDA(h, cudaDeviceGetStreamPriorityRange(&lo, &hi));
  FR_CUDA(h, cudaStreamCreateWithPriority(&h->aux_stream, cudaStreamNonBlocking, hi));
  FR_CUDA(h, cudaEventCreateWithFlags(&h->aux_fork, cudaEventDisableTiming));
  FR_CUDA(h, cudaEventCreateWithFlags(&h->aux_fork2, cudaEventDisableTiming));
  FR_CUDA(h, cudaEventCreateWithFlags(&h->aux_join, cudaEventDisableTiming));
  FR_CUDA(h, cudaStreamCreateWithPriority(&h->aux2_stream, cudaStreamNonBlocking, hi));
  FR_CUDA(h, cudaEventCreateWithFlags(&h->aux2_fork, cudaEventDisableTiming));
  FR_CUDA(h, cudaEventCreateWithFlags(&h->aux2_join, cudaEventDisableTiming));
  return FR_OK;
}

static inline int bits_for(int64_t n) {  // bits needed to represent ids in [0, n)
  int b = 0;
  while (b < 32 && ((int64_t)1 << b) < n) ++b;
  return b < 1 ? 1 : b;
}

static inline int alloc_sort(fr_ctx* h, SortBufs& s, size_t cap) {
  s.cap = (int)cap;
  for (int i = 0; i < 2; ++i) {
    int rc = dalloc(h, &s.k[i], cap); if (rc) return rc;
    rc = dalloc(h, &s.v[i], cap); if (rc) return rc;
  }
  const size_t ntiles = (cap + SORT_TILE - 1) / SORT_TILE;
  int rc = dalloc(h, &s.tile_hist, RADIX_BINS * ntiles + 1); if (rc) return rc;
  if ((rc = dalloc(h, &s.ticket, 1))) return rc;
  FR_CUDA(h, cudaMemset(s.ticket, 0, sizeof(uint32_t)));
  return dalloc(h, &s.scan_tmp, (RADIX_BINS * ntiles) / 4096 + 2);
}


void catalog_free(fr_ctx* h);
// Persisting-L2 access window over [ptr, ptr+bytes) for the kernels queued next on `st` (api.cu)
bool l2_window(fr_ctx* h, const void* ptr, size_t bytes, cudaAccessPolicyWindow* w);
static inline fr::HealthBlend health_of(const fr_ctx* h) {
  fr::HealthBlend hb{nullptr, nullptr, nullptr, 0.f};
  if (h->health_blend) { hb.G = reinterpret_cast<const float4*>(h->tab.G); hb.lab_off = h->tab.user_label_off; hb.lab_idx = h->tab.user_label_idx; hb.alpha = h->mc.alpha; }
  return hb;
}
int ensure_lr_hist(fr_ctx* h, int64_t need, cudaStream_t st);
int shadow_sync(fr_ctx* h, cudaStream_t st);     // rows whose current copy is the shadow go back to the caller's tables
float adam_lr_t(const fr_ctx* h);
fr::OptConsts make_oc(const fr_ctx* h, int64_t step);
// Phases of a training step, shared by fr_train_step and the row-sharded phases (api.cu)
bool single_pass(const fr_ctx* h);              // the step runs the single-pass kernel (lazy Adam, fr_set_shadow)
int tab_code(const fr_ctx* h, bool R_is_table);  // FwdParams::tab
int label_entries(fr_ctx* h, const StepRows& r, const Launch& l);   // label entry list, sorted; returns the sort's result
void label_pass(fr_ctx* h, const StepRows& r, int rl, const Launch& l);
int forward(fr_ctx* h, const StepRows& r, bool fused, const fr::OptConsts& oc, const Launch& l);   // returns its grid
int user_update(fr_ctx* h, const StepRows& r, bool fused, bool write_personal, const fr::OptConsts& oc, int64_t step,
                Launch l, cudaEvent_t before_personal);
void optimizer_tail(fr_ctx* h, const fr::OptConsts& oc, int64_t step, const Launch& l);
void step_advance(fr_ctx* h, int64_t step);
