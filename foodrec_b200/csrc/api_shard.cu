// Row-sharded training step: the five phases declared in include/foodrec_b200.h.  The
// collectives between them belong to the caller (torch.distributed over NCCL/NVLink, or the
// in-process emulation the tests use); nothing here talks to another GPU.
#include "ctx.h"

static int shard_check(fr_ctx* h, const fr_shard* sh) {
  if (!h || !h->has_tables) return fail(h, FR_ERR_STATE, "fr_set_tables first");
  if (!sh || sh->world < 1 || sh->world > 8 || sh->rank < 0 || sh->rank >= sh->world || sh->cap < 1 ||
      sh->items_per_rank < 1 || sh->global_batch < 1)
    return fail(h, FR_ERR_ARG, "bad fr_shard (1 <= world <= 8, cap >= 1)");
  if (sh->items_per_rank != h->cfg.num_items)
    return fail(h, FR_ERR_ARG, "fr_shard.items_per_rank=%d != local Recipe_Embedding rows %d", sh->items_per_rank, h->cfg.num_items);
  return FR_OK;
}

template <class T>
static int ws_alloc(fr_ctx* h, T** p, size_t n) {
  if (*p) { for (auto& q : h->allocs) if (q == *p) { cudaFree(q); q = nullptr; } *p = nullptr; }
  return dalloc(h, p, n);
}

// Buffers of plan slot `idx` for S item rows.  Slot 0 aliases the single-GPU step's workspace (sized max_rows at
// fr_create); slot 1 gets its own on first use.
static int plan_slot_ensure(fr_ctx* h, int idx, size_t S) {
  auto& ps = h->sh.ps[idx];
  int rc;
  if (!ps.owner_counts && (rc = dalloc(h, &ps.owner_counts, 8))) return rc;     // (needed even by a rank with no rows)
  if (!ps.flag_out) {
    if (idx == 0) {
      ps.flag_out = h->out_internal; ps.ukeys = h->ukeys; ps.users_s = h->users_s; ps.items_s = h->items_s; ps.ws_row = h->ws_row;
      ps.sortU = h->sortU; ps.sortI = h->sortI;
      if ((rc = dalloc(h, &ps.scan_tmp, (size_t)h->cfg.max_rows / 4096 + 2))) return rc;   // (h->scan_tmp belongs to forward's label scan)
    } else {
      const size_t M = (size_t)h->cfg.max_rows;
      if ((rc = dalloc(h, &ps.flag_out, FR_OUT_COUNT)) || (rc = dalloc(h, &ps.ukeys, M)) || (rc = dalloc(h, &ps.users_s, M)) ||
          (rc = dalloc(h, &ps.items_s, M)) || (rc = dalloc(h, &ps.ws_row, M)) || (rc = alloc_sort(h, ps.sortU, M)) ||
          (rc = alloc_sort(h, ps.sortI, M)) || (rc = dalloc(h, &ps.scan_tmp, M / 4096 + 2)))
        return rc;
    }
  }
  if (S > ps.s_cap) {
    if (S < (size_t)h->cfg.max_rows) S = (size_t)h->cfg.max_rows;     // once, at capacity: the row count of an un-routed
                                                                      // batch changes every step and a regrow synchronises
    if ((rc = ws_alloc(h, &ps.okeys, S)) || (rc = ws_alloc(h, &ps.flags, S)) || (rc = ws_alloc(h, &ps.excl, S)) ||
        (rc = ws_alloc(h, &ps.slot_sorted, S)) || (rc = ws_alloc(h, &ps.slot_of_row, S)) ||
        (rc = ws_alloc(h, &ps.cats_row, S)))
      return rc;
    ps.s_cap = S;
  }
  return FR_OK;
}

static int owner_ensure(fr_ctx* h, size_t n) {            // owner-side buffers for W*cap request slots
  auto& w = h->sh;
  int rc;
  for (auto& sv : w.ss)
    if (!sv.n_valid && (rc = dalloc(h, &sv.n_valid, 1))) return rc;
  if (!w.route_counts && (rc = dalloc(h, &w.route_counts, 8))) return rc;
  if (n > w.n_cap) {
    for (auto& sv : w.ss) {
      if ((rc = ws_alloc(h, &sv.serve_keys, n))) return rc;
      if ((rc = alloc_sort(h, sv.sortS, n))) return rc;    // (old buffers stay in allocs until fr_destroy)
      sv.prepared = false;
    }
    if ((rc = ws_alloc(h, &w.pieces_s, (n / 32 + 2) * 2 * (size_t)h->mc.DV))) return rc;
    w.n_cap = n;
  }
  return FR_OK;
}

extern "C" int64_t fr_shard_packed_len(fr_handle h) {
  return h ? 4 + 4 * (int64_t)h->mc.D + 5 * (int64_t)h->mc.L * h->mc.D : 0;
}

// ---------------------------------------------------------------- 1. plan
extern "C" int fr_shard_plan(fr_handle h, const fr_batch* b, const fr_shard* sh, int32_t* req, fr_stream s) {
  int rc = shard_check(h, sh); if (rc) return rc;
  if (!b || !req) return fail(h, FR_ERR_ARG, "null batch/req");
  if (b->mode != FR_POINTWISE && b->mode != FR_BPR) return fail(h, FR_ERR_ARG, "bad mode %d", b->mode);
  const int group = b->mode == FR_BPR ? 2 : 1, B = b->n_groups;
  // B == 0 is a first-class case: samples are routed to their user's owner, so with the reference's user-contiguous,
  // unshuffled instance stream (Train_recommender.py:74-96: up to 250 consecutive rows of ONE user) most ranks own no
  // row of a 128-row global batch.  Such a rank requests nothing, contributes zeros to the packed all-reduce, and
  // still serves its peers' requests, applies the replicated Cat / G update and the gradient rows it receives.
  if (B < 0) return fail(h, FR_ERR_ARG, "negative batch size %d", B);
  if ((int64_t)B * group > h->cfg.max_rows) return fail(h, FR_ERR_ARG, "batch exceeds max_rows=%d", h->cfg.max_rows);
  if (B > 0 && (!b->users || !b->items)) return fail(h, FR_ERR_ARG, "users/items are required");
  if (B > 0 && b->mode == FR_POINTWISE && !b->labels) return fail(h, FR_ERR_ARG, "labels are required in pointwise mode");
  if (!b->cats && !h->tab.item_cats) return fail(h, FR_ERR_ARG, "cats is NULL and no (global) item_cats table");
  if (!b->user_labels && !(h->tab.user_label_off && h->tab.user_label_idx))
    return fail(h, FR_ERR_ARG, "user_labels is NULL and no user-label CSR table");
  const int S = B * group, W = sh->world;
  const size_t n = (size_t)W * sh->cap;
  auto& w = h->sh;
  if (w.n_plan - w.n_apply >= 2) return fail(h, FR_ERR_STATE, "fr_shard_plan: both plan slots are in use (plan may run at most one step ahead)");
  const int slot = (int)(w.n_plan & 1);
  if ((rc = plan_slot_ensure(h, slot, (size_t)S)) || (rc = owner_ensure(h, n))) return rc;
  auto& ps = w.ps[slot];
  cudaStream_t st = (cudaStream_t)s;
  const bool lazy_adam = h->cfg.learner == FR_ADAM && h->cfg.adam_mode != FR_ADAM_DENSE;
  if (!(lazy_adam && h->shP) && (rc = shadow_sync(h, st))) return rc;
  Launch l{h->sm_count, st, nullptr};
  ps.mode = b->mode; ps.B = B; ps.S = S; ps.group = group; ps.planned = true; ps.fused = false;
  ++w.n_plan;
  const fr_tables& T = h->tab;
  // (everything written here belongs to the plan slot: this call may overlap the previous step's update / apply.  The
  //  Category_Embedding snapshot and the step counters are taken by fr_shard_forward, after the previous step is done)
  FR_CUDA(h, cudaMemsetAsync(ps.owner_counts, 0, 8 * sizeof(uint32_t), st));
  FR_CUDA(h, cudaMemsetAsync(req, 0xff, n * sizeof(int32_t), st));
  FR_CUDA(h, cudaMemsetAsync(ps.flag_out, 0, FR_OUT_COUNT * sizeof(float), st));
  if (S == 0) return FR_OK;                       // nothing to request: req stays all -1
  // users are LOCAL rows, items GLOBAL recipe ids (< W * items_per_rank; ids in the padding of the last shard are
  // zero rows of their owner): range-checked copies, read by every later phase
  launch_prep_rows(b->mode, B, b->users, b->items, b->labels, b->write_sign, h->cfg.num_users,
                   (int64_t)W * sh->items_per_rank, ps.ukeys, ps.ws_row, ps.users_s, ps.items_s,
                   ps.flag_out + FR_OUT_OVERFLOW, l);

  ShardPlanParams p{};
  p.S = S; p.W = W; p.cap = sh->cap; p.items_per_rank = (uint32_t)sh->items_per_rank;
  p.items = ps.items_s; p.item_cats = (const float4*)T.item_cats; p.cats_in = (const float4*)b->cats;
  p.okeys = ps.okeys; p.cats_row = ps.cats_row;
  p.flags = ps.flags; p.excl = ps.excl; p.owner_counts = ps.owner_counts;
  p.req = req; p.slot_of_row = ps.slot_of_row; p.slot_sorted = ps.slot_sorted; p.out = ps.flag_out;
  launch_shard_prep(p, l);
  SortJob sj[2] = {{&ps.sortU, ps.ukeys, (uint32_t)S, nullptr, bits_for(h->cfg.num_users), 0},
                   {&ps.sortI, ps.okeys, (uint32_t)S, nullptr, bits_for((int64_t)W * sh->items_per_rank), 0}};
  radix_sort_jobs(sj, 2, st, h->sm_count);
  ps.ru = sj[0].result; ps.ri = sj[1].result;
  p.okeys_sorted = ps.sortI.k[ps.ri]; p.perm = ps.sortI.v[ps.ri];
  launch_shard_heads(p, l);
  exclusive_scan_u32(ps.flags, ps.excl, (uint32_t)S, ps.scan_tmp, nullptr, st);
  launch_shard_fill(p, l);
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}

// ---------------------------------------------------------------- routing of an un-routed batch
extern "C" int64_t fr_shard_route_block(const fr_batch* b, int32_t rcap) {
  if (!b || rcap < 1) return 0;
  const int group = b->mode == FR_BPR ? 2 : 1;
  return (int64_t)rcap * (1 + group + (b->mode == FR_POINTWISE ? 1 : 0));
}

extern "C" int fr_shard_route(fr_handle h, const fr_batch* b, int32_t world, int32_t rcap, int32_t* send, float* out_flag,
                              fr_stream s) {
  if (!h) return FR_ERR_ARG;
  if (!b || !send || world < 1 || world > 8 || rcap < 1) return fail(h, FR_ERR_ARG, "bad fr_shard_route arguments");
  if (b->mode != FR_POINTWISE && b->mode != FR_BPR) return fail(h, FR_ERR_ARG, "bad mode %d", b->mode);
  const int B = b->n_groups, group = b->mode == FR_BPR ? 2 : 1;
  if (B < 0 || (int64_t)B * group > h->cfg.max_rows) return fail(h, FR_ERR_ARG, "batch exceeds max_rows=%d", h->cfg.max_rows);
  if (B > 0 && (!b->users || !b->items || (b->mode == FR_POINTWISE && !b->labels))) return fail(h, FR_ERR_ARG, "users/items/labels are required");
  int rc;
  auto& w = h->sh;
  const int slot = (int)(w.n_plan & 1);              // the slot the NEXT fr_shard_plan will use: routing belongs to that step
  if ((rc = plan_slot_ensure(h, slot, (size_t)B * group))) return rc;
  auto& ps = w.ps[slot];
  cudaStream_t st = (cudaStream_t)s;
  Launch l{h->sm_count, st, nullptr};
  const int64_t blk = fr_shard_route_block(b, rcap);
  FR_CUDA(h, cudaMemsetAsync(send, 0xff, (size_t)world * blk * sizeof(int32_t), st));
  FR_CUDA(h, cudaMemsetAsync(ps.owner_counts, 0, 8 * sizeof(uint32_t), st));
  if (B == 0) return FR_OK;
  float* flag = out_flag ? out_flag : ps.flag_out + FR_OUT_OVERFLOW;
  launch_route_keys(b->users, B, world, ps.okeys, ps.owner_counts, l);
  const int r = radix_sort_pairs(ps.sortI, ps.okeys, (uint32_t)B, nullptr, 3, st, h->sm_count);
  launch_route_fill(b->users, b->items, b->mode == FR_POINTWISE ? b->labels : nullptr, B, world, group, rcap, ps.sortI.k[r],
                    ps.sortI.v[r], ps.owner_counts, send, flag, l);
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}

extern "C" int fr_shard_unroute(fr_handle h, int32_t mode, int32_t world, int32_t rcap, const int32_t* recv, int32_t cap_out,
                                int32_t* users, int32_t* items, float* labels, int32_t* n_out, float* out_flag, fr_stream s) {
  if (!h) return FR_ERR_ARG;
  if (!recv || !users || !items || !n_out || world < 1 || world > 8 || rcap < 1 || cap_out < 1) return fail(h, FR_ERR_ARG, "bad fr_shard_unroute arguments");
  if (mode == FR_POINTWISE && !labels) return fail(h, FR_ERR_ARG, "labels buffer required in pointwise mode");
  int rc;
  if ((rc = owner_ensure(h, 0))) return rc;
  cudaStream_t st = (cudaStream_t)s;
  Launch l{h->sm_count, st, nullptr};
  const int group = mode == FR_BPR ? 2 : 1;
  const int blk = rcap * (1 + group + (mode == FR_POINTWISE ? 1 : 0));
  if (!out_flag) return fail(h, FR_ERR_ARG, "fr_shard_unroute needs out_flag");
  float* flag = out_flag;
  launch_route_unpack(recv, world, blk, rcap, group, mode == FR_POINTWISE, h->sh.route_counts, cap_out, users, items, labels,
                      n_out, flag, l);
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}

extern "C" int fr_gather_user_rows(fr_handle h, const int32_t* users, int32_t n, float* out, fr_stream s) {
  if (!h || !h->has_tables) return fail(h, FR_ERR_STATE, "fr_set_tables first");
  if (n < 0 || (n > 0 && (!users || !out))) return fail(h, FR_ERR_ARG, "null argument");
  if (n == 0) return FR_OK;
  cudaStream_t st = (cudaStream_t)s;
  int rc = shadow_sync(h, st); if (rc) return rc;
  Launch l{h->sm_count, st, nullptr};
  PeerPtrs none{}; none.world = 0;
  launch_gather_rows((const float4*)h->tab.P, users, (uint32_t)n, 5 * h->mc.DV, (float4*)out, none, l, (uint32_t)h->cfg.num_users,
                     h->table_bf16 ? 1 : 0);
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}

// ---------------------------------------------------------------- peer-memory exchange
extern "C" int fr_shard_set_peers(fr_handle h, const fr_shard* sh, float* const* peer_rbuf, float* const* peer_rgrows) {
  int rc = shard_check(h, sh); if (rc) return rc;
  if (!peer_rbuf || !peer_rgrows) return fail(h, FR_ERR_ARG, "null peer table");
  auto& w = h->sh;
  for (int r = 0; r < sh->world; ++r) {
    if (!peer_rbuf[r] || !peer_rgrows[r]) return fail(h, FR_ERR_ARG, "null peer buffer for rank %d", r);
    w.peer_rbuf.dst[r] = reinterpret_cast<float4*>(peer_rbuf[r]);
    w.peer_rgrows.dst[r] = reinterpret_cast<float4*>(peer_rgrows[r]);
  }
  w.peer_rbuf.world = w.peer_rgrows.world = sh->world;
  w.peer_rbuf.rank = w.peer_rgrows.rank = sh->rank;
  w.peer_rbuf.cap = w.peer_rgrows.cap = sh->cap;
  return FR_OK;
}

// ---------------------------------------------------------------- 2. serve
// received requests -> (recipe, slot) keys, stable sort by recipe: the order the catch-up and fr_shard_apply walk.
// Depends on the request list only, not on the tables.
static void serve_sort(fr_ctx* h, const fr_shard* sh, const int32_t* rreq, fr_ctx::ShardWs::ServeSlot& sv, size_t n, const Launch& l) {
  launch_serve_keys(rreq, (uint32_t)n, (uint32_t)sh->items_per_rank, sv.serve_keys, sv.n_valid, l);
  sv.rs = radix_sort_pairs(sv.sortS, sv.serve_keys, (uint32_t)n, nullptr, bits_for((int64_t)sh->items_per_rank + 1), l.st, h->sm_count);
  sv.prepared = true;
}

extern "C" int fr_shard_serve_prepare(fr_handle h, const fr_shard* sh, const int32_t* rreq, fr_stream s) {
  int rc = shard_check(h, sh); if (rc) return rc;
  if (!rreq) return fail(h, FR_ERR_ARG, "null rreq");
  auto& w = h->sh;
  if (w.n_plan <= w.n_apply) return fail(h, FR_ERR_STATE, "fr_shard_plan must precede fr_shard_serve_prepare");
  const size_t n = (size_t)sh->world * sh->cap;
  if ((rc = owner_ensure(h, n))) return rc;
  Launch l{h->sm_count, (cudaStream_t)s, nullptr};
  serve_sort(h, sh, rreq, w.ss[(w.n_plan - 1) & 1], n, l);     // the step planned last
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}

extern "C" int fr_shard_serve(fr_handle h, const fr_shard* sh, const int32_t* rreq, float* rows, fr_stream s) {
  int rc = shard_check(h, sh); if (rc) return rc;
  if (!rreq) return fail(h, FR_ERR_ARG, "null rreq");
  if (!rows && h->sh.peer_rbuf.world != sh->world) return fail(h, FR_ERR_ARG, "rows is NULL but fr_shard_set_peers has not been called for this world");
  const size_t n = (size_t)sh->world * sh->cap;
  if ((rc = owner_ensure(h, n))) return rc;
  cudaStream_t st = (cudaStream_t)s;
  Launch l{h->sm_count, st, nullptr};
  auto& w = h->sh;
  const fr_tables& T = h->tab;
  const int64_t step = h->step + 1;
  if ((rc = ensure_lr_hist(h, step + 1, st))) return rc;
  const OptConsts oc = make_oc(h, step);
  auto& sv = w.ss[w.n_apply & 1];
  if (!sv.prepared) serve_sort(h, sh, rreq, sv, n, l);      // (else fr_shard_serve_prepare did it, one step ahead)
  if (h->cfg.learner == FR_ADAM && h->cfg.adam_mode != FR_ADAM_DENSE)    // requested rows must be current
    launch_item_catchup(h->NV, sv.sortS.k[sv.rs], (uint32_t)n, (float4*)T.R, (float4*)T.s1_R, (float4*)T.s2_R, T.last_R,
                        h->mc.DV, oc, l, sv.n_valid);
  PeerPtrs none{}; none.world = 0;
  launch_gather_rows((const float4*)T.R, rreq, (uint32_t)n, h->mc.DV, (float4*)rows, rows ? none : w.peer_rbuf, l,
                     (uint32_t)h->cfg.num_items, h->table_bf16 ? 1 : 0);
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}

// ---------------------------------------------------------------- 3. forward
// The rows of this rank's step (plan slot ps), read from the received recipe rows
static StepRows shard_rows(fr_ctx* h, const fr_ctx::PlanSlot& ps, const fr_batch* b, const fr_shard* sh, const float* rbuf,
                           float* out, float* dG) {
  StepRows r{};
  r.B = ps.B; r.S = ps.S; r.group = ps.group;
  r.users = ps.users_s; r.items = ps.slot_of_row; r.ws_row = ps.ws_row;
  r.ukeys = ps.sortU.k[ps.ru]; r.uperm = ps.sortU.v[ps.ru];
  r.R = (const float4*)rbuf; r.R_is_table = false; r.cats = ps.cats_row; r.cats_by_item = 0;
  r.labels = b->labels; r.user_labels = b->user_labels; r.Bnorm = (float)sh->global_batch;
  r.out = out; r.scores = h->scores; r.G = (float4*)dG;
  return r;
}

extern "C" int fr_shard_forward(fr_handle h, const fr_batch* b, const fr_shard* sh, const float* rbuf, float* packed,
                                fr_stream s) {
  int rc = shard_check(h, sh); if (rc) return rc;
  if (!b || !rbuf || !packed) return fail(h, FR_ERR_ARG, "null argument");
  auto& w = h->sh;
  auto& ps = w.ps[w.n_apply & 1];
  if (!ps.planned || b->n_groups != ps.B) return fail(h, FR_ERR_STATE, "fr_shard_plan must precede fr_shard_forward");
  cudaStream_t st = (cudaStream_t)s;
  FR_CUDA(h, cudaMemsetAsync(h->counters, 0, 4 * sizeof(uint32_t), st));
  if (ps.S == 0) {     // a rank without rows adds nothing to {loss, sum|g|^2, dCat, dG}
    FR_CUDA(h, cudaMemsetAsync(packed, 0, (size_t)fr_shard_packed_len(h) * sizeof(float), st));
    ps.fused = false;
    return FR_OK;
  }
  // pre-step snapshot of Category_Embedding (every read of Cat in this step sees it)
  FR_CUDA(h, cudaMemcpyAsync(h->cat_pre, h->tab.Cat, (size_t)4 * h->mc.D * sizeof(float), cudaMemcpyDeviceToDevice, st));
  Launch l{h->sm_count, st, nullptr};
  const OptConsts oc = make_oc(h, h->step + 1);
  const StepRows r = shard_rows(h, ps, b, sh, rbuf, ps.flag_out, packed + 4 + 4 * (size_t)h->mc.D);

  // General_Memory delta of this rank's rows -> packed (G itself is updated after the all-reduce).  Entry list and segment
  // reduce read only the batch, the received rows and the Cat snapshot: they run on the library's side stream BESIDE the
  // forward / single-pass kernel (bandwidth-bound; this chain is issue- and latency-bound), joined at the end of the phase.
  if ((rc = aux_ensure(h))) return rc;
  FR_CUDA(h, cudaEventRecord(h->aux_fork, st));
  FR_CUDA(h, cudaStreamWaitEvent(h->aux_stream, h->aux_fork, 0));
  const Launch la{h->sm_count, h->aux_stream, nullptr};
  FR_CUDA(h, cudaMemsetAsync(r.G, 0, 5 * (size_t)h->mc.L * h->mc.D * sizeof(float), la.st));
  label_pass(h, r, label_entries(h, r, la), la);
  FR_CHECK_LAUNCH(h);
  FR_CUDA(h, cudaEventRecord(h->aux_join, h->aux_stream));

  // single-pass: forward AND the speculative Personal_Memory update, before the all-reduce that makes the global norm
  // known; fr_shard_update commits the rows (scale == 1) or redoes the update with the true scale
  ps.fused = single_pass(h);
  const int fgrid = forward(h, r, ps.fused, oc, l);
  FinalizeParams fin{};
  fin.part_loss = h->part_loss; fin.part_nrm = h->part_nrm; fin.part_gcat = h->part_gcat; fin.nblk = fgrid;
  fin.DV = h->mc.DV; fin.B = r.Bnorm; fin.packed = packed; fin.do_reduce = 1; fin.do_apply = 0;
  fin.oc = oc; fin.clip = h->cfg.clip_norm; fin.out = ps.flag_out; fin.lr_hist = nullptr;
  launch_finalize(fin, l);
  FR_CUDA(h, cudaStreamWaitEvent(st, h->aux_join, 0));
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}

// ---------------------------------------------------------------- 4. update
extern "C" int fr_shard_update(fr_handle h, const fr_batch* b, const fr_shard* sh, int32_t write_personal,
                               const float* rbuf, const float* packed_reduced, float* grows, float* out_scalars,
                               fr_stream s) {
  int rc = shard_check(h, sh); if (rc) return rc;
  if (!b || !rbuf || !packed_reduced) return fail(h, FR_ERR_ARG, "null argument");
  auto& w = h->sh;
  auto& ps = w.ps[w.n_apply & 1];
  if (!grows && w.peer_rgrows.world != sh->world) return fail(h, FR_ERR_ARG, "grows is NULL but fr_shard_set_peers has not been called for this world");
  if (h->table_bf16 && write_personal) return fail(h, FR_ERR_UNSUPPORTED, "personal-write steps are not available with bf16 tables");
  if (!ps.planned || b->n_groups != ps.B) return fail(h, FR_ERR_STATE, "fr_shard_plan must precede fr_shard_update");
  cudaStream_t st = (cudaStream_t)s;
  Launch l{h->sm_count, st, nullptr};
  const fr_tables& T = h->tab;
  const int DV = h->mc.DV, NV = h->NV, S = ps.S;
  const int64_t step = h->step + 1;
  const OptConsts oc = make_oc(h, step);
  float* out = out_scalars ? out_scalars : ps.flag_out;
  if (out != ps.flag_out)   // flags raised by plan/forward (capacity / label overflow / id range)
    FR_CUDA(h, cudaMemcpyAsync(out, ps.flag_out, FR_OUT_COUNT * sizeof(float), cudaMemcpyDeviceToDevice, st));
  const StepRows r = shard_rows(h, ps, b, sh, rbuf, out, nullptr);

  // fr_timing_*: the events of this phase's kernels (user pass, personal pass + dG add as "label", local recipe-gradient
  // pass); the phases that live in other fr_shard_* calls read as zero
  const StepTiming tm(h, st);
  tm.mark(FR_T_SORT); tm.mark(FR_T_FWD); tm.mark(FR_T_FINALIZE);
  FinalizeParams fin{};
  fin.DV = DV; fin.B = r.Bnorm; fin.packed = const_cast<float*>(packed_reduced);
  fin.do_reduce = 0; fin.do_apply = 1;
  fin.Cat = (float4*)T.Cat; fin.s1Cat = (float4*)T.s1_Cat; fin.s2Cat = (float4*)T.s2_Cat;
  fin.oc = oc; fin.clip = h->cfg.clip_norm; fin.out = out; fin.lr_hist = h->lr_hist;
  launch_finalize(fin, l);

  tm.mark(FR_T_USER_CHUNK);
  l.mid = tm.ev(FR_T_USER_COMBINE);
  if ((rc = user_update(h, r, ps.fused, write_personal, oc, step, l, tm.ev(FR_T_LABEL)))) return rc;
  l.mid = nullptr;
  // G += all-reduced delta (after the personal pass, which reads G_old)
  launch_add_inplace((float4*)T.G, (const float4*)(packed_reduced + 4 + 4 * (size_t)h->mc.D), (int64_t)h->mc.L * 5 * DV, l);

  // finished gradient rows of the recipes this rank touched, in the owners' slot order
  SegCommon ci{};
  ci.keys = ps.slot_sorted; ci.perm = ps.sortI.v[ps.ri]; ci.n_dev = nullptr; ci.n_host = (uint32_t)S;
  ci.pieces = h->pieces_i; ci.uniq_counter = h->counters + 1;
  ci.long_list = h->long_list; ci.long_count = h->counters + 3; ci.long_cap = h->long_cap;
  ItemPolParams ip{};
  ip.z = h->z; ip.g = h->g; ip.out = out; ip.mc = h->mc; ip.oc = oc;
  PeerPtrs none{}; none.world = 0;
  tm.mark(FR_T_ITEM_CHUNK);
  l.mid = tm.ev(FR_T_ITEM_COMBINE);
  if (S > 0) launch_item_grad_pass(NV, ci, ip, (float4*)grows, grows ? none : w.peer_rgrows, l);
  else if (l.mid) cudaEventRecord(l.mid, st);
  l.mid = nullptr;
  tm.mark(FR_T_SWEEP); tm.mark(FR_T_MISC); tm.mark(FR_T_COUNT);
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}

// ---------------------------------------------------------------- 5. apply
extern "C" int fr_shard_apply(fr_handle h, const fr_shard* sh, const int32_t* rreq, const float* rgrows,
                              float* out_scalars, fr_stream s) {
  int rc = shard_check(h, sh); if (rc) return rc;
  if (!rreq || !rgrows) return fail(h, FR_ERR_ARG, "null argument");
  auto& w = h->sh;
  auto& ps = w.ps[w.n_apply & 1];
  if (!ps.planned) return fail(h, FR_ERR_STATE, "fr_shard_plan must precede fr_shard_apply");
  cudaStream_t st = (cudaStream_t)s;
  Launch l{h->sm_count, st, nullptr};
  const fr_tables& T = h->tab;
  const int DV = h->mc.DV, NV = h->NV;
  const int64_t step = h->step + 1;
  const OptConsts oc = make_oc(h, step);
  float* out = out_scalars ? out_scalars : ps.flag_out;
  const uint32_t n = (uint32_t)((size_t)sh->world * sh->cap);

  // received (recipe, gradient row) pairs, sorted by recipe at serve time (stable: rank order)
  SegCommon c{};
  auto& sv = w.ss[w.n_apply & 1];
  if (!sv.prepared) return fail(h, FR_ERR_STATE, "fr_shard_serve must precede fr_shard_apply");
  c.keys = sv.sortS.k[sv.rs]; c.perm = sv.sortS.v[sv.rs]; c.n_dev = sv.n_valid; c.n_host = n;
  c.pieces = w.pieces_s; c.uniq_counter = nullptr;
  ItemPolParams ip{};
  ip.R = (float4*)T.R; ip.s1 = (float4*)T.s1_R; ip.s2 = (float4*)T.s2_R; ip.last = T.last_R;
  ip.z = (const float4*)rgrows; ip.g = nullptr; ip.out = out; ip.mc = h->mc; ip.oc = oc; ip.tab = tab_code(h, true);
  launch_item_pass(NV, c, ip, l);
  optimizer_tail(h, oc, step, l);
  launch_mean((const float4*)T.G, (int64_t)h->mc.L * 5 * DV, h->mean_partials, out + FR_OUT_GENERAL,
              (double)h->mc.L * 5.0 * h->mc.D, l);
  launch_write_counters(h->counters, out, l);
  FR_CHECK_LAUNCH(h);
  ps.S = 0; ps.planned = false;
  sv.prepared = false;
  ++w.n_apply;
  step_advance(h, step);
  return FR_OK;
}
