// C ABI of libfoodrec_b200.so (see include/foodrec_b200.h): context, workspace and the
// orchestration of one training step.  No compute happens on the host; there is no CPU
// fallback -- every entry point fails with FR_ERR_CUDA if the device is unusable.
#include "ctx.h"

extern "C" int fr_abi_version(void) { return FR_ABI_VERSION; }

extern "C" int fr_create(const fr_config* cfg, fr_handle* out) {
  if (!cfg || !out) return FR_ERR_ARG;
  *out = nullptr;
  fr_ctx* h = new fr_ctx();
  *out = h;   // returned even on failure so fr_last_error works; caller must fr_destroy
  h->cfg = *cfg;
  const int D = cfg->embed_size;
  if (D <= 0 || D % 4 != 0 || D > 256) return fail(h, FR_ERR_ARG, "embed_size must be a multiple of 4 in (0,256], got %d", D);
  if (cfg->num_users <= 0 || cfg->num_items <= 0 || cfg->num_labels <= 0 || cfg->max_rows <= 0)
    return fail(h, FR_ERR_ARG, "num_users/num_items/num_labels/max_rows must be positive");
  if (cfg->learner < FR_SGD || cfg->learner > FR_ADAM) return fail(h, FR_ERR_ARG, "bad learner %d", cfg->learner);
  if (cfg->learner == FR_ADAM && cfg->adam_mode == FR_ADAM_LAZY_SERIES) {
    // The closed-form catch-up keeps SERIES_TERMS terms over a window of SERIES_WINDOW steps; both are sized for
    // the TF default betas.  For the configured betas: the skipped tail b1^WINDOW must be negligible and the
    // truncated terms  sum_j b1^j d_j^5 / (1 - d_j),  d_j = 1 - b2^(j/2),  must stay below fp32 round-off of the
    // leading term  sum_j b1^j -- otherwise rows that sat out many steps would be caught up wrongly, silently.
    const double b1 = cfg->adam_beta1, b2 = cfg->adam_beta2;
    if (!(b1 >= 0.0 && b1 < 1.0 && b2 > 0.0 && b2 < 1.0)) return fail(h, FR_ERR_ARG, "adam betas must lie in [0,1) / (0,1)");
    double lead = 0.0, rem = 0.0, p1 = 1.0;
    for (int j = 1; j <= SERIES_WINDOW; ++j) {
      p1 *= b1;
      const double d = 1.0 - pow(b2, 0.5 * j);
      lead += p1;
      rem += p1 * pow(d, SERIES_TERMS) / (1.0 - d);
    }
    if (p1 > 1e-12 || (lead > 0.0 && rem / lead > 1e-7))
      return fail(h, FR_ERR_UNSUPPORTED, "adam_mode LAZY_SERIES does not cover beta1=%g beta2=%g (tail %.1e, truncation %.1e): "
                  "use FR_ADAM_LAZY_EXACT", b1, b2, p1, lead > 0.0 ? rem / lead : 0.0);
  }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(h, FR_ERR_CUDA, "no CUDA device (%s); foodrec_b200 has no CPU fallback", cudaGetErrorString(e));
  FR_CUDA(h, cudaGetDevice(&h->device));
  cudaDeviceProp prop;
  FR_CUDA(h, cudaGetDeviceProperties(&prop, h->device));
  h->sm_count = prop.multiProcessorCount;
  h->l2_persist_max = (size_t)prop.persistingL2CacheMaxSize;
  h->l2_window_max = (size_t)prop.accessPolicyMaxWindowSize;
  if (getenv("FOODREC_NO_L2_PIN")) h->l2_persist_max = 0;
  if (getenv("FOODREC_DEBUG_L2"))
    fprintf(stderr, "foodrec_b200: L2 %d MB, persisting max %zu MB, access window max %zu MB\n", prop.l2CacheSize >> 20,
            h->l2_persist_max >> 20, h->l2_window_max >> 20);
  h->mc.D = D; h->mc.DV = D / 4; h->mc.L = cfg->num_labels;
  h->mc.a = cfg->high_level_score_coefficient;
  h->mc.oma = 1.0f - cfg->high_level_score_coefficient;     // fp32 (1 - a), Model_Recommender.py:96
  h->mc.beta_1 = cfg->beta_1; h->mc.beta_2 = cfg->beta_2; h->mc.alpha = cfg->alpha;
  h->NV = h->mc.DV <= 32 ? 1 : 2;
  h->b1p = cfg->adam_beta1; h->b2p = cfg->adam_beta2;

  const size_t S = (size_t)cfg->max_rows, E = (size_t)(cfg->max_label_entries > 0 ? cfg->max_label_entries : 1);
  const size_t DV = h->mc.DV;
  int rc;
#define A(p, n) if ((rc = dalloc(h, &(p), (n)))) return rc
  A(h->ukeys, S); A(h->users_s, S); A(h->items_s, S); A(h->ws_row, S); A(h->g, S); A(h->scores, S); A(h->z, S * DV);
  if ((rc = alloc_sort(h, h->sortU, S))) return rc;
  if ((rc = alloc_sort(h, h->sortI, S))) return rc;
  if ((rc = alloc_sort(h, h->sortL, E))) return rc;
  h->fwd_grid_cap = h->sm_count * 4;
  A(h->part_loss, h->fwd_grid_cap); A(h->part_nrm, h->fwd_grid_cap); A(h->part_gcat, (size_t)h->fwd_grid_cap * 4 * DV);
  A(h->packed, 4 + 4 * (size_t)D + 5 * (size_t)cfg->num_labels * D);   // loss, |g|^2, dCat (+ dG when sharded)
  const size_t chS = S / 32 + 2, chE = E / 32 + 2;
  A(h->pieces_u, chS * 2 * 5 * DV); A(h->pieces_i, chS * 2 * DV); A(h->pieces_g, chE * 2 * 5 * DV);
  h->long_cap = (uint32_t)((chS > chE ? chS : chE) / FR_LONG_CHAIN + 2);
  A(h->long_list, h->long_cap);
  A(h->counts, S + 1); A(h->offs, S + 1); A(h->ent_key, E); A(h->ent_row, E); A(h->ent_coef, E); A(h->n_entries, 1);
  A(h->counters, 4); A(h->cat_pre, 4 * DV); A(h->mean_partials, 1024); A(h->out_internal, FR_OUT_COUNT);
  A(h->scan_tmp, S / 4096 + 2);
  h->lr_hist_cap = 1 << 16;
  A(h->lr_hist, (size_t)h->lr_hist_cap);
  A(h->cser, (size_t)h->lr_hist_cap * SERIES_TERMS);
#undef A
  FR_CUDA(h, cudaMemset(h->lr_hist, 0, (size_t)h->lr_hist_cap * sizeof(float)));
  FR_CUDA(h, cudaMemset(h->cser, 0, (size_t)h->lr_hist_cap * SERIES_TERMS * sizeof(double)));
  FR_CUDA(h, cudaMemset(h->out_internal, 0, FR_OUT_COUNT * sizeof(float)));
  return FR_OK;
}

extern "C" int64_t fr_launch_count(void) { return (int64_t)fr::g_launches; }

// A table that every work item of a kernel re-reads at random (Recipe_Embedding in sampled evaluation: 51 rows per
// user) should stay in L2 while a much larger read-once stream (the user rows) passes through it.  A persisting
// access-policy window on the table marks its lines persisting; if the table is larger than the persisting carve-out
// (79 MB of B200's 126 MB L2; the cfg2 recipe table is 102 MB), hitRatio pins that fraction of it.
bool l2_window(fr_ctx* h, const void* ptr, size_t bytes, cudaAccessPolicyWindow* w) {
  if (!h->l2_persist_max || !h->l2_window_max || !bytes) return false;
  static bool limit_set = false;
  if (!limit_set) { cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, h->l2_persist_max); cudaGetLastError(); limit_set = true; }
  const size_t win = bytes < h->l2_window_max ? bytes : h->l2_window_max;
  w->base_ptr = const_cast<void*>(ptr);
  w->num_bytes = win;
  const double r = (double)h->l2_persist_max / (double)win;
  w->hitRatio = r >= 1.0 ? 1.0f : (float)r;
  w->hitProp = cudaAccessPropertyPersisting;
  w->missProp = cudaAccessPropertyNormal;      // the part of the window beyond the carve-out is cached as usual (Streaming
                                               // would turn that fraction of the table's reads into certain misses)
  return true;
}

extern "C" int fr_timing_enable(fr_handle h, int32_t enable) {
  if (!h) return FR_ERR_ARG;
  if (enable && h->tsets.empty()) {
    h->tsets.resize(32);
    for (auto& ts : h->tsets)
      for (auto& e : ts.ev) FR_CUDA(h, cudaEventCreate(&e));
  }
  h->timing = enable != 0;
  return FR_OK;
}

extern "C" int fr_timing_read(fr_handle h, double* ms_sum, int64_t* n_steps, int32_t reset) {
  if (!h || !ms_sum || !n_steps) return FR_ERR_ARG;
  for (auto& ts : h->tsets) timing_collect(h, ts);
  for (int i = 0; i < FR_T_COUNT; ++i) ms_sum[i] = h->t_sum[i];
  *n_steps = h->t_steps;
  if (reset) { for (auto& x : h->t_sum) x = 0.0; h->t_steps = 0; }
  return FR_OK;
}

extern "C" int fr_destroy(fr_handle h) {
  if (!h) return FR_OK;
  for (auto& ts : h->tsets) for (auto& e : ts.ev) cudaEventDestroy(e);
  catalog_free(h);
  for (void* p : h->allocs) cudaFree(p);
  if (h->stage) cudaFree(h->stage);
  for (auto& sl : h->feed) { if (sl.buf) cudaFree(sl.buf); if (sl.copied) cudaEventDestroy(sl.copied); if (sl.consumed) cudaEventDestroy(sl.consumed); }
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->aux_stream) { cudaStreamDestroy(h->aux_stream); cudaEventDestroy(h->aux_fork); cudaEventDestroy(h->aux_fork2); cudaEventDestroy(h->aux_join);
                       cudaStreamDestroy(h->aux2_stream); cudaEventDestroy(h->aux2_fork); cudaEventDestroy(h->aux2_join); }
  if (h->pieces_personal) cudaFree(h->pieces_personal);
  delete h;
  return FR_OK;
}

extern "C" const char* fr_last_error(fr_handle h) { return h ? h->err : "null handle"; }

extern "C" int fr_set_tables(fr_handle h, const fr_tables* t) {
  if (!h || !t) return FR_ERR_ARG;
  if (!t->P || !t->R || !t->Cat || !t->G) return fail(h, FR_ERR_ARG, "P/R/Cat/G must be non-null");
  const int L = h->cfg.learner;
  if (L != FR_SGD && (!t->s1_P || !t->s1_R || !t->s1_Cat)) return fail(h, FR_ERR_ARG, "optimizer slot s1 missing");
  if ((L == FR_ADAM || L == FR_RMSPROP) && (!t->s2_P || !t->s2_R || !t->s2_Cat)) return fail(h, FR_ERR_ARG, "optimizer slot s2 missing");
  if (L == FR_ADAM && (!t->last_P || !t->last_R)) return fail(h, FR_ERR_ARG, "Adam needs last_P/last_R stamps");
  const uintptr_t al = (uintptr_t)t->P | (uintptr_t)t->R | (uintptr_t)t->Cat | (uintptr_t)t->G |
                       (uintptr_t)t->s1_P | (uintptr_t)t->s2_P | (uintptr_t)t->s1_R | (uintptr_t)t->s2_R |
                       (uintptr_t)t->s1_Cat | (uintptr_t)t->s2_Cat | (uintptr_t)t->item_cats;
  if (al & 15) return fail(h, FR_ERR_ARG, "table pointers must be 16-byte aligned");
  h->tab = *t;
  h->has_tables = true;
  return FR_OK;
}

extern "C" int fr_set_table_format(fr_handle h, int32_t format) {
  if (!h) return FR_ERR_ARG;
  if (format != FR_TABLE_F32 && format != FR_TABLE_BF16) return fail(h, FR_ERR_ARG, "unknown table format %d", format);
  if (h->has_tables) return fail(h, FR_ERR_STATE, "fr_set_table_format must precede fr_set_tables");
  if (format == FR_TABLE_BF16 && h->cfg.learner == FR_ADAM)
    return fail(h, FR_ERR_UNSUPPORTED, "bf16 tables are offered for SGD / Adagrad / RMSProp: TF-1.x Adam moves every row every "
                "step, which re-rounds all of Personal_Memory to bf16 each time (see include/foodrec_b200.h)");
  h->table_bf16 = format == FR_TABLE_BF16;
  return FR_OK;
}

extern "C" int fr_set_shadow(fr_handle h, float* P_alt, float* s1_alt, float* s2_alt) {
  if (!h || !h->has_tables) return fail(h, FR_ERR_STATE, "fr_set_tables first");
  if (h->table_bf16 && (P_alt || s1_alt || s2_alt)) return fail(h, FR_ERR_UNSUPPORTED, "the single-pass step is not available with bf16 tables");
  if (!P_alt && !s1_alt && !s2_alt) {             // switch the single-pass step off again
    int rc = shadow_sync(h, 0); if (rc) return rc;
    FR_CUDA(h, cudaDeviceSynchronize());
    h->shP = h->shM = h->shV = nullptr;
    return FR_OK;
  }
  if (h->cfg.learner != FR_ADAM || h->cfg.adam_mode == FR_ADAM_DENSE)
    return fail(h, FR_ERR_UNSUPPORTED, "the single-pass step exists for lazy Adam only (FR_ADAM with FR_ADAM_LAZY_*)");
  if (!P_alt || !s1_alt || !s2_alt) return fail(h, FR_ERR_ARG, "all three shadow tables are required");
  if (((uintptr_t)P_alt | (uintptr_t)s1_alt | (uintptr_t)s2_alt) & 15) return fail(h, FR_ERR_ARG, "shadow tables must be 16-byte aligned");
  if ((int64_t)h->cfg.num_users >= (int64_t)FR_SHADOW_BIT) return fail(h, FR_ERR_UNSUPPORTED, "too many rows");
  h->shP = P_alt; h->shM = s1_alt; h->shV = s2_alt;
  return FR_OK;
}

int shadow_sync(fr_ctx* h, cudaStream_t st) {
  if (!h->shadow_dirty || !h->shP) return FR_OK;
  Launch l{h->sm_count, st, nullptr};
  launch_shadow_consolidate(h->tab.last_P, h->cfg.num_users, 5 * h->mc.DV, (float4*)h->tab.P, (float4*)h->tab.s1_P,
                            (float4*)h->tab.s2_P, (const float4*)h->shP, (const float4*)h->shM, (const float4*)h->shV,
                            nullptr, l);
  FR_CHECK_LAUNCH(h);
  h->shadow_dirty = false;
  return FR_OK;
}

extern "C" int fr_get_step(fr_handle h, int64_t* step) {
  if (!h || !step) return FR_ERR_ARG;
  *step = h->step;
  return FR_OK;
}

int ensure_lr_hist(fr_ctx* h, int64_t need, cudaStream_t st) {
  if (need < h->lr_hist_cap) return FR_OK;
  int64_t cap = h->lr_hist_cap;
  while (cap <= need) cap *= 2;
  float* nb = nullptr;
  double* nc = nullptr;
  const size_t cb_old = (size_t)h->lr_hist_cap * SERIES_TERMS * sizeof(double), cb_new = (size_t)cap * SERIES_TERMS * sizeof(double);
  FR_CUDA(h, cudaMalloc(&nb, (size_t)cap * sizeof(float)));
  FR_CUDA(h, cudaMalloc(&nc, cb_new));
  FR_CUDA(h, cudaMemsetAsync(nb, 0, (size_t)cap * sizeof(float), st));
  FR_CUDA(h, cudaMemsetAsync(nc, 0, cb_new, st));
  FR_CUDA(h, cudaMemcpyAsync(nb, h->lr_hist, (size_t)h->lr_hist_cap * sizeof(float), cudaMemcpyDeviceToDevice, st));
  FR_CUDA(h, cudaMemcpyAsync(nc, h->cser, cb_old, cudaMemcpyDeviceToDevice, st));
  FR_CUDA(h, cudaStreamSynchronize(st));
  for (auto& p : h->allocs) { if (p == h->lr_hist) p = nb; else if (p == h->cser) p = nc; }
  cudaFree(h->lr_hist); cudaFree(h->cser);
  h->lr_hist = nb; h->cser = nc; h->lr_hist_cap = cap;
  return FR_OK;
}

float adam_lr_t(const fr_ctx* h) {   // adam.py: lr * sqrt(1 - beta2_power) / (1 - beta1_power), fp32
  const float num = h->cfg.lr * sqrtf(1.0f - h->b2p);
  return num / (1.0f - h->b1p);
}

extern "C" int fr_set_step(fr_handle h, int64_t step) {
  if (!h || step < 0) return FR_ERR_ARG;
  int rc = ensure_lr_hist(h, step + 1, 0); if (rc) return rc;
  std::vector<float> hist((size_t)step + 1, 0.f);
  h->b1p = h->cfg.adam_beta1; h->b2p = h->cfg.adam_beta2;
  for (int64_t t = 1; t <= step; ++t) {
    hist[(size_t)t] = adam_lr_t(h);
    h->b1p *= h->cfg.adam_beta1; h->b2p *= h->cfg.adam_beta2;
  }
  FR_CUDA(h, cudaMemcpy(h->lr_hist, hist.data(), hist.size() * sizeof(float), cudaMemcpyHostToDevice));
  FR_CUDA(h, cudaMemset(h->cser, 0, (size_t)h->lr_hist_cap * SERIES_TERMS * sizeof(double)));
  if (h->cfg.learner == FR_ADAM && h->cfg.adam_mode == FR_ADAM_LAZY_SERIES) {
    Launch l{h->sm_count, 0, nullptr};
    launch_series_rebuild(h->cser, h->lr_hist, (int)step, h->cfg.adam_beta1, h->cfg.adam_beta2, l);
    FR_CUDA(h, cudaDeviceSynchronize());
  }
  h->step = step;
  return FR_OK;
}

OptConsts make_oc(const fr_ctx* h, int64_t step) {
  OptConsts oc{};
  oc.learner = h->cfg.learner; oc.adam_mode = h->cfg.adam_mode;
  oc.lr = h->cfg.lr; oc.lr_t = adam_lr_t(h);
  oc.b1 = h->cfg.adam_beta1; oc.b2 = h->cfg.adam_beta2; oc.eps = h->cfg.adam_eps;
  oc.omb1 = 1.0f - oc.b1; oc.omb2 = 1.0f - oc.b2;
  oc.rho = h->cfg.rms_decay; oc.omrho = 1.0f - oc.rho; oc.rms_eps = h->cfg.rms_eps;
  oc.step = (int)step; oc.lr_hist = h->lr_hist;
  oc.cser = h->cser; oc.l2b1 = log2f(oc.b1); oc.l2b2 = log2f(oc.b2);
  return oc;
}

extern "C" int fr_set_health_blend(fr_handle h, int32_t enable) {
  if (!h) return FR_ERR_ARG;
  if (enable && (!h->has_tables || !h->tab.user_label_off || !h->tab.user_label_idx))
    return fail(h, FR_ERR_STATE, "the health term needs the resident user-label CSR (tables.user_label_off/idx)");
  h->health_blend = enable != 0;
  return FR_OK;
}

extern "C" int fr_fwd_score(fr_handle h, const int32_t* users, const int32_t* items, const float* cats,
                            int32_t n, float* scores, fr_stream s) {
  if (!h || !h->has_tables) return fail(h, FR_ERR_STATE, "fr_set_tables first");
  if (n < 0 || (n > 0 && (!users || !items || !scores))) return fail(h, FR_ERR_ARG, "null batch pointer");
  if (!cats && !h->tab.item_cats) return fail(h, FR_ERR_ARG, "cats is NULL and no item_cats table");
  { int rc = shadow_sync(h, (cudaStream_t)s); if (rc) return rc; }
  Launch l{h->sm_count, (cudaStream_t)s};
  launch_fwd_score(h->mc, (const float4*)h->tab.P, (const float4*)h->tab.R, (const float4*)h->tab.Cat, users, items,
                   (const float4*)(cats ? cats : h->tab.item_cats), cats ? 0 : 1, n, scores, health_of(h), l,
                   h->cfg.num_users, h->cfg.num_items, h->table_bf16 ? 1 : 0);
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}

extern "C" int fr_eval_sampled_topk(fr_handle h, const int32_t* users, const int32_t* cand, const int32_t* n_cand,
                                    int32_t n_users, int32_t cand_stride, const float* cand_cats, int32_t K,
                                    int32_t* topk_ids, int32_t* gt_rank, float* scores, fr_stream s) {
  if (!h || !h->has_tables) return fail(h, FR_ERR_STATE, "fr_set_tables first");
  if (n_users < 0 || cand_stride <= 0 || cand_stride > 128 || K <= 0) return fail(h, FR_ERR_ARG, "need 0<cand_stride<=128, K>0");
  if (n_users > 0 && (!users || !cand || !n_cand || !topk_ids || !gt_rank)) return fail(h, FR_ERR_ARG, "null pointer");
  if (!cand_cats && !h->tab.item_cats) return fail(h, FR_ERR_ARG, "cand_cats is NULL and no item_cats table");
  if ((int64_t)h->cfg.num_items * h->mc.DV >= (1ll << 32))     // (row offsets travel between lanes as 32-bit words)
    return fail(h, FR_ERR_UNSUPPORTED, "fr_eval_sampled_topk: Recipe_Embedding of %d x %d exceeds 2^32 16-byte groups", h->cfg.num_items, h->mc.D);
  { int rc = shadow_sync(h, (cudaStream_t)s); if (rc) return rc; }
  Launch l{h->sm_count, (cudaStream_t)s};
  cudaAccessPolicyWindow win{};
  if (l2_window(h, h->tab.R, (size_t)h->cfg.num_items * h->mc.D * sizeof(float), &win)) { l.win = &win; h->l2_lines_pinned = true; }
  launch_eval_sampled(h->mc, (const float4*)h->tab.P, (const float4*)h->tab.R, (const float4*)h->tab.Cat, users, cand,
                      n_cand, n_users, cand_stride, (const float4*)cand_cats, (const float4*)h->tab.item_cats, K,
                      topk_ids, gt_rank, scores, health_of(h), l, h->cfg.num_users, h->cfg.num_items, h->table_bf16 ? 1 : 0);
  // (lines the window marked persisting are demoted by cudaCtxResetPersistingL2Cache at the next fr_train_step)
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}

extern "C" int fr_sort_pairs(fr_handle h, const uint32_t* keys, int32_t n, int32_t nbits, uint32_t* out_keys,
                             uint32_t* out_idx, fr_stream s) {
  if (!h) return FR_ERR_ARG;
  if (n < 0 || n > h->sortU.cap) return fail(h, FR_ERR_ARG, "n=%d exceeds max_rows=%d", n, h->sortU.cap);
  if (n == 0) return FR_OK;
  cudaStream_t st = (cudaStream_t)s;
  const int r = radix_sort_pairs(h->sortU, keys, (uint32_t)n, nullptr, nbits, st, h->sm_count);
  FR_CHECK_LAUNCH(h);
  FR_CUDA(h, cudaMemcpyAsync(out_keys, h->sortU.k[r], (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
  FR_CUDA(h, cudaMemcpyAsync(out_idx, h->sortU.v[r], (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
  return FR_OK;
}

extern "C" int fr_adam_flush(fr_handle h, fr_stream s) {
  if (!h || !h->has_tables) return fail(h, FR_ERR_STATE, "fr_set_tables first");
  { int rc = shadow_sync(h, (cudaStream_t)s); if (rc) return rc; }
  if (h->cfg.learner != FR_ADAM || h->step == 0) return FR_OK;
  Launch l{h->sm_count, (cudaStream_t)s};
  const OptConsts oc = make_oc(h, h->step);
  launch_adam_sweep((float4*)h->tab.P, (float4*)h->tab.s1_P, (float4*)h->tab.s2_P, h->tab.last_P, h->cfg.num_users,
                    5 * h->mc.DV, oc, (int)h->step, l);
  launch_adam_sweep((float4*)h->tab.R, (float4*)h->tab.s1_R, (float4*)h->tab.s2_R, h->tab.last_R, h->cfg.num_items,
                    h->mc.DV, oc, (int)h->step, l);
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}

// ---------------------------------------------------------------- phases of a training step
// Built once for both callers: fr_train_step reads the tables, fr_shard_forward / fr_shard_update the rows this rank
// planned and received (StepRows).  Launch errors are left for the caller's FR_CHECK_LAUNCH.

// The single-pass step: forward + Personal_Memory update in one kernel on the double-buffered table (train_seg.cu)
bool single_pass(const fr_ctx* h) {
  return h->cfg.learner == FR_ADAM && h->cfg.adam_mode != FR_ADAM_DENSE && h->shP && !getenv("FOODREC_TWO_PASS");
}

// Storage of the tables a pass reads: 0 fp32 P and R, 1 bf16 P and R, 2 bf16 P + fp32 R (received rows).  The passes
// that read only recipe rows (LabelPolParams, ItemPolParams) read bf16 ones for code 1 alone.
int tab_code(const fr_ctx* h, bool R_is_table) { return !h->table_bf16 ? 0 : R_is_table ? 1 : 2; }

// Entry list of the General_Memory pass: non-zeros of the label feed -> (label, row, coef), sorted by label
int label_entries(fr_ctx* h, const StepRows& r, const Launch& l) {
  LabelEmitParams ep{};
  ep.S = r.S; ep.group = r.group; ep.L = h->mc.L; ep.users = r.users;
  ep.user_labels = r.user_labels; ep.lab_off = h->tab.user_label_off; ep.lab_idx = h->tab.user_label_idx;
  ep.ws_row = r.ws_row; ep.counts = h->counts; ep.offs = h->offs;
  ep.ent_key = h->ent_key; ep.ent_row = h->ent_row; ep.ent_coef = h->ent_coef;
  ep.cap = (uint32_t)h->sortL.cap; ep.n_entries = h->n_entries; ep.out = r.out;
  launch_label_count(ep, l);
  exclusive_scan_u32(h->counts, h->offs, (uint32_t)r.S, h->scan_tmp, h->n_entries, l.st);
  launch_label_emit(ep, l);
  return radix_sort_pairs(h->sortL, h->ent_key, ep.cap, h->n_entries, bits_for(h->mc.L), l.st, h->sm_count);
}

// General_Memory: segment reduce of the label entries (sort result rl) by label into r.G.  It reads pre-step state only.
// (Round 2 tried a shared-memory scatter with one owner warp per label instead -- no sort, no entry list: measured
// 354 us + 25 us against this pass's 254 us at 524k rows; see DESIGN.md "measured and rejected".)
void label_pass(fr_ctx* h, const StepRows& r, int rl, const Launch& l) {
  SegCommon c{};
  c.keys = h->sortL.k[rl]; c.perm = h->sortL.v[rl]; c.n_dev = h->n_entries; c.n_host = (uint32_t)h->sortL.cap;
  c.pieces = h->pieces_g; c.uniq_counter = nullptr;
  c.long_list = h->long_list; c.long_count = h->counters + 2; c.long_cap = h->long_cap;
  LabelPolParams lp{};
  lp.G = r.G; lp.R = r.R; lp.cat = h->cat_pre;
  lp.ent_row = h->ent_row; lp.ent_coef = h->ent_coef; lp.items = r.items; lp.cats = r.cats;
  lp.cats_by_item = r.cats_by_item; lp.mc = h->mc; lp.tab = tab_code(h, r.R_is_table) == 1;
  launch_label_pass(h->NV, c, lp, l);
}

static SegCommon user_seg(fr_ctx* h, const StepRows& r) {   // the rows by user
  SegCommon c{};
  c.keys = r.ukeys; c.perm = r.uperm; c.n_dev = nullptr; c.n_host = (uint32_t)r.S;
  c.uniq_counter = h->counters + 0; c.pieces = h->pieces_u;
  return c;
}

// Forward, loss, per-slice norms, dCat partials, z stash.  Single-pass (fused): also the segment reduce by user and Adam
// with the clip scale speculated = 1, new rows into the other copy of the double-buffered Personal_Memory; user_update
// commits them once the norm is known.  l.mid: recorded between the single-pass kernel and its crossing-run combine.
// Returns the grid, whose per-block partials finalize reduces.
int forward(fr_ctx* h, const StepRows& r, bool fused, const OptConsts& oc, const Launch& l) {
  const fr_tables& T = h->tab;
  if (fused) {
    FusedParams fz{};
    fz.P[0] = (float4*)T.P; fz.m[0] = (float4*)T.s1_P; fz.v[0] = (float4*)T.s2_P;
    fz.P[1] = (float4*)h->shP; fz.m[1] = (float4*)h->shM; fz.v[1] = (float4*)h->shV;
    fz.last = T.last_P; fz.R = r.R; fz.cat = h->cat_pre;
    fz.items = r.items; fz.cats = r.cats; fz.cats_by_item = r.cats_by_item; fz.labels = r.labels;
    fz.a = h->mc.a; fz.oma = h->mc.oma; fz.Bnorm = r.Bnorm;
    fz.g = h->g; fz.z = h->z; fz.scores = r.scores;
    fz.part_loss = h->part_loss; fz.part_nrm = h->part_nrm; fz.part_gcat = h->part_gcat;
    fz.mc = h->mc; fz.oc = oc;
    const int grid = user_fused_grid((uint32_t)r.S, h->sm_count);
    launch_user_fused(h->NV, r.group, user_seg(h, r), fz, grid, l);
    h->shadow_dirty = true;
    return grid;
  }
  FwdParams fp{};
  fp.P = (const float4*)T.P; fp.R = r.R; fp.cat = h->cat_pre; fp.DV = h->mc.DV; fp.B = r.B; fp.Bnorm = r.Bnorm;
  fp.users = r.users; fp.items = r.items; fp.cats = r.cats; fp.cats_by_item = r.cats_by_item;
  fp.labels = r.labels; fp.a = h->mc.a; fp.oma = h->mc.oma;
  fp.g = h->g; fp.z = h->z; fp.scores = r.scores;
  fp.part_loss = h->part_loss; fp.part_nrm = h->part_nrm; fp.part_gcat = h->part_gcat;
  fp.lazy = h->cfg.learner == FR_ADAM && h->cfg.adam_mode != FR_ADAM_DENSE;
  fp.mP = (const float4*)T.s1_P; fp.vP = (const float4*)T.s2_P; fp.lastP = T.last_P; fp.oc = oc;
  fp.tab = tab_code(h, r.R_is_table);
  const int grid = fwd_train_grid(r.B, h->sm_count);
  launch_fwd_train(h->NV, r.group, fp, grid, l);
  return grid;
}

// Personal_Memory: segment reduce by user + optimizer, then on personal steps Write_Memory (Model_Recommender.py:149-198)
// on the optimizer's output, which reads pre-step R, Cat, G.  l.mid: recorded between the user pass's chunk kernel and
// its combine; before_personal (nullable): recorded after the user pass.
int user_update(fr_ctx* h, const StepRows& r, bool fused, bool write_personal, const OptConsts& oc, int64_t step,
                Launch l, cudaEvent_t before_personal) {
  const fr_tables& T = h->tab;
  SegCommon c = user_seg(h, r);
  UserPolParams up{};
  up.P = (float4*)T.P; up.s1 = (float4*)T.s1_P; up.s2 = (float4*)T.s2_P; up.last = T.last_P;
  up.R = r.R; up.G = (const float4*)T.G; up.cat = h->cat_pre;
  up.items = r.items; up.g = h->g; up.cats = r.cats; up.cats_by_item = r.cats_by_item;
  up.ws_row = r.ws_row; up.out = r.out; up.group = r.group; up.mc = h->mc; up.oc = oc;
  up.user_labels = r.user_labels; up.lab_off = T.user_label_off; up.lab_idx = T.user_label_idx; up.users = r.users;
  up.tab = tab_code(h, r.R_is_table);
  if (r.S == 0) {
    if (l.mid) cudaEventRecord(l.mid, l.st);
  } else {
    if (fused) {
      // the norm is known.  scale == 1 exactly: the speculative rows become current (stamp bits flipped).  Otherwise
      // nothing was committed: every row goes back to the caller's tables and the ordinary update pass runs with the
      // true scale on the g / z the single-pass kernel left (both launches exit at once in the common case).
      launch_user_commit(c.keys, (uint32_t)r.S, T.last_P, r.out, (int)step, l);
      launch_shadow_consolidate(T.last_P, h->cfg.num_users, 5 * h->mc.DV, (float4*)T.P, (float4*)T.s1_P,
                                (float4*)T.s2_P, (const float4*)h->shP, (const float4*)h->shM, (const float4*)h->shV,
                                r.out, l);
      c.uniq_counter = nullptr;          // (counted by the single-pass kernel)
      c.only_if_scaled = r.out;
    }
    launch_user_pass(h->NV, c, up, l);
  }
  l.mid = nullptr;
  if (before_personal) cudaEventRecord(before_personal, l.st);
  if (!write_personal || r.S == 0) return FR_OK;
  if (fused) { int rc = shadow_sync(h, l.st); if (rc) return rc; }     // the personal pass works on the caller's table
  c.only_if_scaled = nullptr;                                         // (it always runs, whatever the clip did)
  const size_t need = (size_t)r.S / 32 + 2;
  if (need > h->pieces_personal_chunks) {
    if (h->pieces_personal) { FR_CUDA(h, cudaStreamSynchronize(l.st)); cudaFree(h->pieces_personal); h->pieces_personal = nullptr; }
    FR_CUDA(h, cudaMalloc(&h->pieces_personal, need * 2 * 10 * h->mc.DV * sizeof(float4)));
    h->pieces_personal_chunks = need;
  }
  c.pieces = h->pieces_personal; c.uniq_counter = nullptr;
  launch_personal_pass(h->NV, c, up, l);
  return FR_OK;
}

// LAZY_SERIES table: every catch-up of this step (target t-1) is done; add the s = t term so that the table serves
// target t (a personal step's sweep, fr_adam_flush, step t+1).  TF-1.x dense Adam: every untouched row decays this step too.
void optimizer_tail(fr_ctx* h, const OptConsts& oc, int64_t step, const Launch& l) {
  const fr_tables& T = h->tab;
  if (h->cfg.learner == FR_ADAM && h->cfg.adam_mode == FR_ADAM_LAZY_SERIES)
    launch_series_update(h->cser, h->lr_hist, (int)step, h->cfg.adam_beta1, h->cfg.adam_beta2, l);
  if (h->cfg.learner == FR_ADAM && h->cfg.adam_mode == FR_ADAM_DENSE) {
    launch_adam_sweep((float4*)T.P, (float4*)T.s1_P, (float4*)T.s2_P, T.last_P, h->cfg.num_users, 5 * h->mc.DV, oc, (int)step, l);
    launch_adam_sweep((float4*)T.R, (float4*)T.s1_R, (float4*)T.s2_R, T.last_R, h->cfg.num_items, h->mc.DV, oc, (int)step, l);
  }
}

void step_advance(fr_ctx* h, int64_t step) {
  h->step = step;
  h->b1p *= h->cfg.adam_beta1;     // adam.py _finish
  h->b2p *= h->cfg.adam_beta2;
}

extern "C" int fr_train_step(fr_handle h, const fr_batch* b, int32_t write_personal, float* out_scalars,
                             float* out_scores, fr_stream s) {
  if (!h || !h->has_tables) return fail(h, FR_ERR_STATE, "fr_set_tables first");
  if (!b) return fail(h, FR_ERR_ARG, "null batch");
  if (b->mode != FR_POINTWISE && b->mode != FR_BPR) return fail(h, FR_ERR_ARG, "bad mode %d", b->mode);
  const int group = b->mode == FR_BPR ? 2 : 1;
  const int B = b->n_groups;
  const int64_t S64 = (int64_t)B * group;
  if (B <= 0) return fail(h, FR_ERR_ARG, "empty batch (n_groups=%d): the reference never runs one "
                                         "(Train_recommender.py:163-166 drops the tail)", B);
  if (S64 > h->cfg.max_rows) return fail(h, FR_ERR_ARG, "batch has %lld item rows > max_rows=%d", (long long)S64, h->cfg.max_rows);
  const int S = (int)S64;
  if (!b->users || !b->items) return fail(h, FR_ERR_ARG, "users/items are required");
  if (b->mode == FR_POINTWISE && !b->labels) return fail(h, FR_ERR_ARG, "labels are required in pointwise mode");
  if (!b->cats && !h->tab.item_cats) return fail(h, FR_ERR_ARG, "cats is NULL and no item_cats table");
  if (!b->user_labels && !(h->tab.user_label_off && h->tab.user_label_idx))
    return fail(h, FR_ERR_ARG, "user_labels is NULL and no user-label CSR table");
  if (h->table_bf16 && write_personal) return fail(h, FR_ERR_UNSUPPORTED, "personal-write steps are not available with bf16 tables");
  cudaStream_t st = (cudaStream_t)s;
  if (h->l2_lines_pinned) { cudaCtxResetPersistingL2Cache(); cudaGetLastError(); h->l2_lines_pinned = false; }
  Launch l{h->sm_count, st, nullptr};
  const fr_tables& T = h->tab;
  const int DV = h->mc.DV, NV = h->NV;
  const int64_t step = h->step + 1;
  int rc = ensure_lr_hist(h, step + 1, st); if (rc) return rc;
  const OptConsts oc = make_oc(h, step);
  float* out = out_scalars ? out_scalars : h->out_internal;
  StepRows r{};
  r.B = B; r.S = S; r.group = group;
  r.users = h->users_s; r.items = h->items_s; r.ws_row = h->ws_row;     // range-checked: every kernel below reads these
  r.R = (const float4*)T.R; r.R_is_table = true;
  r.cats = (const float4*)(b->cats ? b->cats : T.item_cats); r.cats_by_item = b->cats ? 0 : 1;
  r.labels = b->labels; r.user_labels = b->user_labels; r.Bnorm = (float)B;
  r.out = out; r.scores = out_scores ? out_scores : h->scores; r.G = (float4*)T.G;

  const StepTiming tm(h, st);
  tm.mark(FR_T_SORT);
  // 0. pre-step snapshot of Category_Embedding (every read of Cat in this step sees it)
  FR_CUDA(h, cudaMemcpyAsync(h->cat_pre, T.Cat, (size_t)4 * h->mc.D * sizeof(float), cudaMemcpyDeviceToDevice, st));
  FR_CUDA(h, cudaMemsetAsync(h->counters, 0, 4 * sizeof(uint32_t), st));
  FR_CUDA(h, cudaMemsetAsync(out + FR_OUT_OVERFLOW, 0, sizeof(float), st));

  // 1. row keys, write sign; sort item rows by user and by recipe
  launch_prep_rows(b->mode, B, b->users, b->items, b->labels, b->write_sign, h->cfg.num_users, h->cfg.num_items, h->ukeys,
                   h->ws_row, h->users_s, h->items_s, out + FR_OUT_OVERFLOW, l);
  // 1b. FORK: the General_Memory pass's entry list depends only on the batch.  It is ~0.1 ms of small latency-bound
  //     kernels (count, scan, emit, one radix pass) that used to sit on the step's critical path; they now run on a side
  //     stream beside the sorts / catch-up / forward (which are small or bandwidth-bound) and are joined before the label
  //     segment-reduce needs them.
  if ((rc = aux_ensure(h))) return rc;
  FR_CUDA(h, cudaEventRecord(h->aux_fork, st));
  FR_CUDA(h, cudaStreamWaitEvent(h->aux_stream, h->aux_fork, 0));
  const Launch la{h->sm_count, h->aux_stream, nullptr};
  const int rl = label_entries(h, r, la);
  FR_CHECK_LAUNCH(h);
  SortJob sj[2] = {{&h->sortU, h->ukeys, (uint32_t)S, nullptr, bits_for(h->cfg.num_users), 0},
                   {&h->sortI, (const uint32_t*)h->items_s, (uint32_t)S, nullptr, bits_for(h->cfg.num_items), 0}};
  radix_sort_jobs(sj, 2, st, h->sm_count);      // by user and by recipe, sharing their launches
  const int ri = sj[1].result;
  r.ukeys = h->sortU.k[sj[0].result]; r.uperm = h->sortU.v[sj[0].result];
  FR_CHECK_LAUNCH(h);
  // Personal-write steps (16 per run of the reference, Train_recommender.py:169-187) take the two-pass path.
  const bool fused = single_pass(h) && !write_personal;
  if (!fused) { rc = shadow_sync(h, st); if (rc) return rc; }
  const bool lazy = h->cfg.learner == FR_ADAM && h->cfg.adam_mode != FR_ADAM_DENSE;
  if (lazy) {   // recipe rows of this batch must be current before anything reads them
    launch_item_catchup(NV, h->sortI.k[ri], (uint32_t)S, (float4*)T.R, (float4*)T.s1_R, (float4*)T.s2_R,
                        T.last_R, DV, oc, l);
    FR_CHECK_LAUNCH(h);
  }
  // 1c. General_Memory pass (5): it reads only pre-step state (R rows of this batch -- current after the catch-up above --
  //     the Category_Embedding snapshot, the entry list of 1b) and writes G, which nothing else in the step reads except
  //     a personal-write pass (pre-step G, Model_Recommender.py:170-198) and the final mean.  So on ordinary steps it runs
  //     on the side stream too, beside the forward / user pass (bandwidth-bound; this pass is issue-bound), and is joined
  //     before the recipe pass overwrites R.
  //     (With fr_timing_enable the pass runs in sequence, so that every phase time is that of its kernels alone.)
  const bool label_aside = !write_personal && !h->timing;
  if (label_aside) {
    FR_CUDA(h, cudaEventRecord(h->aux_fork2, st));
    FR_CUDA(h, cudaStreamWaitEvent(h->aux_stream, h->aux_fork2, 0));
    label_pass(h, r, rl, la);
    // the `general` fetch = mean(G) (:219) only needs the pass above: off the main stream too
    launch_mean((const float4*)T.G, (int64_t)h->mc.L * 5 * DV, h->mean_partials, out + FR_OUT_GENERAL,
                (double)h->mc.L * 5.0 * h->mc.D, la);
    FR_CHECK_LAUNCH(h);
  }
  FR_CUDA(h, cudaEventRecord(h->aux_join, h->aux_stream));

  tm.mark(FR_T_FWD);
  // 2. forward.  (Single-pass: the norm / loss / dCat partials are complete when the kernel ends; its crossing-run combine
  //    does not touch them: finalize runs beside the combine on a second side stream -- the event is recorded between the
  //    two launches.  With fr_timing_enable it runs in sequence.)
  const bool fin_aside = fused && !h->timing;
  l.mid = fin_aside ? h->aux2_fork : nullptr;
  const int fgrid = forward(h, r, fused, oc, l);
  l.mid = nullptr;
  FR_CHECK_LAUNCH(h);

  tm.mark(FR_T_FINALIZE);
  // 3. global norm -> clip scale; dense optimizer on Cat
  FinalizeParams fin{};
  fin.part_loss = h->part_loss; fin.part_nrm = h->part_nrm; fin.part_gcat = h->part_gcat; fin.nblk = fgrid;
  fin.DV = DV; fin.B = (float)B; fin.packed = h->packed; fin.do_reduce = 1; fin.do_apply = 1;
  fin.Cat = (float4*)T.Cat; fin.s1Cat = (float4*)T.s1_Cat; fin.s2Cat = (float4*)T.s2_Cat;
  fin.oc = oc; fin.clip = h->cfg.clip_norm; fin.out = out; fin.lr_hist = h->lr_hist;
  if (fin_aside) {
    FR_CUDA(h, cudaStreamWaitEvent(h->aux2_stream, h->aux2_fork, 0));
    launch_finalize(fin, Launch{h->sm_count, h->aux2_stream, nullptr});
    FR_CUDA(h, cudaEventRecord(h->aux2_join, h->aux2_stream));
    FR_CUDA(h, cudaStreamWaitEvent(st, h->aux2_join, 0));
  } else {
    launch_finalize(fin, l);
  }
  FR_CHECK_LAUNCH(h);

  tm.mark(FR_T_USER_CHUNK);
  // 4. Personal_Memory: segment-reduce by user + optimizer (+ personal write)
  l.mid = tm.ev(FR_T_USER_COMBINE);
  if ((rc = user_update(h, r, fused, write_personal, oc, step, l, nullptr))) return rc;
  FR_CHECK_LAUNCH(h);

  tm.mark(FR_T_LABEL);
  // 5. General_Memory (built in 1b, run in 1c on ordinary steps)
  l.mid = nullptr;
  FR_CUDA(h, cudaStreamWaitEvent(st, h->aux_join, 0));      // JOIN: the side stream (entry list 1b, and the pass itself 1c)
  if (!label_aside) { label_pass(h, r, rl, l); FR_CHECK_LAUNCH(h); }

  tm.mark(FR_T_ITEM_CHUNK);
  // 6. Recipe_Embedding: segment-reduce by recipe + optimizer
  {
    l.mid = tm.ev(FR_T_ITEM_COMBINE);
    SegCommon c{};
    c.keys = h->sortI.k[ri]; c.perm = h->sortI.v[ri]; c.n_dev = nullptr; c.n_host = (uint32_t)S;
    c.pieces = h->pieces_i; c.uniq_counter = h->counters + 1;
    c.long_list = h->long_list; c.long_count = h->counters + 3; c.long_cap = h->long_cap;
    ItemPolParams ip{};
    ip.R = (float4*)T.R; ip.s1 = (float4*)T.s1_R; ip.s2 = (float4*)T.s2_R; ip.last = T.last_R;
    ip.z = h->z; ip.g = h->g; ip.out = out; ip.mc = h->mc; ip.oc = oc; ip.tab = tab_code(h, true);
    launch_item_pass(NV, c, ip, l);
    FR_CHECK_LAUNCH(h);
  }

  l.mid = nullptr;
  tm.mark(FR_T_SWEEP);
  optimizer_tail(h, oc, step, l);
  FR_CHECK_LAUNCH(h);

  tm.mark(FR_T_MISC);
  // 8. fetches: general = mean(G) (:219), personal = mean(P) (:218, personal steps only)
  if (!label_aside)
    launch_mean((const float4*)T.G, (int64_t)h->mc.L * 5 * DV, h->mean_partials, out + FR_OUT_GENERAL,
                (double)h->mc.L * 5.0 * h->mc.D, l);
  if (write_personal) {
    if (lazy) {
      // mean(P) must see every row at step t
      launch_adam_sweep((float4*)T.P, (float4*)T.s1_P, (float4*)T.s2_P, T.last_P, h->cfg.num_users, 5 * DV, oc, (int)step, l);
    }
    launch_mean((const float4*)T.P, (int64_t)h->cfg.num_users * 5 * DV, h->mean_partials, out + FR_OUT_PERSONAL,
                (double)h->cfg.num_users * 5.0 * h->mc.D, l);
  }
  launch_write_counters(h->counters, out, l);
  FR_CHECK_LAUNCH(h);
  tm.mark(FR_T_COUNT);
  step_advance(h, step);
  return FR_OK;
}

// byte layout of a batch image in a staging buffer
struct FeedLayout { size_t users, items, cats, labels, ws, ul, out, total; int group; size_t S; };
static FeedLayout feed_layout(const fr_ctx* h, const fr_batch* hb) {
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  FeedLayout f;
  f.group = hb->mode == FR_BPR ? 2 : 1;
  const size_t B = (size_t)hb->n_groups, L = (size_t)h->mc.L;
  f.S = B * f.group;
  f.users = 0;
  f.items = f.users + al(B * 4);
  f.cats = f.items + al(f.S * 4);
  f.labels = f.cats + al(hb->cats ? f.S * 16 : 0);
  f.ws = f.labels + al(hb->labels ? B * 4 : 0);
  f.ul = f.ws + al(hb->write_sign ? f.S * 4 : 0);
  f.out = f.ul + al(hb->user_labels ? B * L * 4 : 0);
  f.total = f.out + al(FR_OUT_COUNT * 4);
  return f;
}
static int feed_copy(fr_ctx* h, const fr_batch* hb, const FeedLayout& f, char* base, fr_batch* db, cudaStream_t st) {
  const size_t B = (size_t)hb->n_groups, L = (size_t)h->mc.L;
  *db = *hb;
#define H2D(field, off, bytes) if (hb->field) { \
    FR_CUDA(h, cudaMemcpyAsync(base + (off), hb->field, (bytes), cudaMemcpyHostToDevice, st)); \
    db->field = reinterpret_cast<decltype(db->field)>(base + (off)); }
  H2D(users, f.users, B * 4)
  H2D(items, f.items, f.S * 4)
  H2D(cats, f.cats, f.S * 16)
  H2D(labels, f.labels, B * 4)
  H2D(write_sign, f.ws, f.S * 4)
  H2D(user_labels, f.ul, B * L * 4)
#undef H2D
  return FR_OK;
}

extern "C" int fr_feed_prefetch(fr_handle h, const fr_batch* hb) {
  if (!h || !hb) return FR_ERR_ARG;
  if (hb->n_groups <= 0) return fail(h, FR_ERR_ARG, "empty batch");
  if (!h->copy_stream) {
    FR_CUDA(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    for (auto& sl : h->feed) {
      FR_CUDA(h, cudaEventCreateWithFlags(&sl.copied, cudaEventDisableTiming));
      FR_CUDA(h, cudaEventCreateWithFlags(&sl.consumed, cudaEventDisableTiming));
    }
  }
  fr_ctx::FeedSlot& sl = h->feed[h->feed_next];
  h->feed_next ^= 1;
  const FeedLayout f = feed_layout(h, hb);
  if (sl.used) FR_CUDA(h, cudaStreamWaitEvent(h->copy_stream, sl.consumed, 0));   // the step that read this slot is done
  if (f.total > sl.bytes) {
    if (sl.buf) { FR_CUDA(h, cudaDeviceSynchronize()); cudaFree(sl.buf); sl.buf = nullptr; }
    FR_CUDA(h, cudaMalloc(&sl.buf, f.total));
    sl.bytes = f.total;
  }
  int rc = feed_copy(h, hb, f, static_cast<char*>(sl.buf), &sl.dev, h->copy_stream);
  if (rc) return rc;
  sl.dout = reinterpret_cast<float*>(static_cast<char*>(sl.buf) + f.out);
  FR_CUDA(h, cudaEventRecord(sl.copied, h->copy_stream));
  sl.host = *hb;
  sl.valid = true;
  return FR_OK;
}

static bool same_batch(const fr_batch& a, const fr_batch& b) {
  return a.mode == b.mode && a.n_groups == b.n_groups && a.users == b.users && a.items == b.items && a.cats == b.cats &&
         a.labels == b.labels && a.write_sign == b.write_sign && a.user_labels == b.user_labels;
}

extern "C" int fr_train_step_host(fr_handle h, const fr_batch* hb, int32_t write_personal,
                                  float* host_out_scalars, fr_stream s) {
  if (!h || !hb) return FR_ERR_ARG;
  for (auto& sl : h->feed) {
    if (sl.valid && same_batch(sl.host, *hb)) {          // staged by fr_feed_prefetch: only wait for its copy
      cudaStream_t st = (cudaStream_t)s;
      FR_CUDA(h, cudaStreamWaitEvent(st, sl.copied, 0));
      sl.valid = false;
      int rc = fr_train_step(h, &sl.dev, write_personal, sl.dout, nullptr, s);
      if (rc) return rc;
      if (host_out_scalars)
        FR_CUDA(h, cudaMemcpyAsync(host_out_scalars, sl.dout, FR_OUT_COUNT * sizeof(float), cudaMemcpyDeviceToHost, st));
      FR_CUDA(h, cudaEventRecord(sl.consumed, st));
      sl.used = true;
      return FR_OK;
    }
  }
  if (hb->n_groups <= 0) return fail(h, FR_ERR_ARG, "empty batch");
  cudaStream_t st = (cudaStream_t)s;
  const FeedLayout f = feed_layout(h, hb);
  if (f.total > h->stage_bytes) {
    if (h->stage) { FR_CUDA(h, cudaStreamSynchronize(st)); cudaFree(h->stage); h->stage = nullptr; }
    FR_CUDA(h, cudaMalloc(&h->stage, f.total));
    h->stage_bytes = f.total;
  }
  fr_batch db;
  int rc = feed_copy(h, hb, f, static_cast<char*>(h->stage), &db, st);
  if (rc) return rc;
  float* dout = reinterpret_cast<float*>(static_cast<char*>(h->stage) + f.out);
  rc = fr_train_step(h, &db, write_personal, dout, nullptr, s);
  if (rc) return rc;
  if (host_out_scalars)
    FR_CUDA(h, cudaMemcpyAsync(host_out_scalars, dout, FR_OUT_COUNT * sizeof(float), cudaMemcpyDeviceToHost, st));
  return FR_OK;
}
