// Sampled evaluation (evaluate.py:35-66) on row-sharded tables.  A test user lives on rank u % W, its candidates are
// GLOBAL recipe ids, recipe i lives on rank i % W at local row i / W.  The user owner
//   fr_shard_eval_plan     dedups its candidates per owner -> req[W*cap] (the training step's request layout) and
//                          rewrites every candidate as a SLOT of the received-row buffer (owner o's k-th smallest
//                          requested row -> o*cap + k), with the slot -> global id map
//     all_to_all(req)
//   fr_shard_eval_serve    owner: the requested rows in the table's own format (fp32, or bf16 as stored)
//     all_to_all(rows)
//   fr_eval_sampled_rows   eval_sampled_kernel unchanged on (Personal_Memory, received rows, slots), then the top-K
//                          slots back to global ids.
// The kernel uses a candidate id only for equality (dict dedup, the held-out item's rank), bounds and addressing; ties
// go to insertion position, not to the id.  Distinct ids get distinct slots and repeats the same slot, so the ranking
// is the one the unsharded engine computes on the global ids.
#include "ctx.h"

namespace fr {

struct EvalPlanParams {
  const int32_t* cand; const int32_t* n_cand;
  uint32_t N; int stride, W; uint32_t ipr, n_items, cap;
  const float4* item_cats; float4* cats_out;         // cats_out [n, stride] (nullable): masks by global id
  uint32_t* keys;                                     // owner-major keys, invalid = W * ipr (sorts last)
  const uint32_t* keys_sorted; const uint32_t* perm;
  uint32_t *flags, *excl, *owner_counts;
  int32_t *req, *slots, *slot_ids;
  float* flag;
};

// one entry per (user, j): valid iff j < n_cand and 0 <= id < n_items (the global catalog, which excludes the padding
// rows of the last recipe shard)
__global__ void eval_plan_keys_kernel(const EvalPlanParams p) {
  const uint32_t bad = (uint32_t)p.W * p.ipr;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < p.N; i += gridDim.x * blockDim.x) {
    const uint32_t w = i / (uint32_t)p.stride, j = i - w * (uint32_t)p.stride;
    const int nc = p.n_cand[w];
    const int32_t id = p.cand[i];
    const bool ok = (int)j < nc && id >= 0 && (uint32_t)id < p.n_items;
    p.keys[i] = ok ? ((uint32_t)id % (uint32_t)p.W) * p.ipr + (uint32_t)id / (uint32_t)p.W : bad;
    if (p.cats_out) p.cats_out[i] = ok ? __ldg(p.item_cats + id) : make_float4(1.f, 0.f, 0.f, 0.f);
  }
}

__global__ void eval_plan_heads_kernel(const EvalPlanParams p) {
  const uint32_t bad = (uint32_t)p.W * p.ipr;
  for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < p.N; q += gridDim.x * blockDim.x) {
    const uint32_t k = p.keys_sorted[q];
    const bool head = k < bad && (q == 0 || p.keys_sorted[q - 1] != k);
    p.flags[q] = head ? 1u : 0u;
    if (head) atomicAdd(p.owner_counts + k / p.ipr, 1u);          // integer: order-independent
  }
}

// unique recipe k (rank of its run) of owner o -> slot o*cap + (k - start[o]); more than cap for one owner raises the
// flag and drops the candidate (never a write past the buffers)
__global__ void eval_plan_fill_kernel(const EvalPlanParams p) {
  const uint32_t bad = (uint32_t)p.W * p.ipr;
  uint32_t start[9];
  start[0] = 0;
  for (int o = 0; o < p.W && o < 8; ++o) start[o + 1] = start[o] + p.owner_counts[o];
  for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < p.N; q += gridDim.x * blockDim.x) {
    const uint32_t key = p.keys_sorted[q], dst = p.perm[q];
    if (key >= bad) { p.slots[dst] = -1; continue; }
    const uint32_t o = key / p.ipr, row = key - o * p.ipr;
    const uint32_t j = p.excl[q] + p.flags[q] - 1u - start[o];
    if (j >= p.cap) { *p.flag = 2.f; p.slots[dst] = -1; continue; }
    const uint32_t slot = o * p.cap + j;
    if (p.flags[q]) { p.req[slot] = (int32_t)row; p.slot_ids[slot] = (int32_t)(row * (uint32_t)p.W + o); }
    p.slots[dst] = (int32_t)slot;
  }
}

__global__ void eval_unslot_kernel(int32_t* __restrict__ ids, size_t n, const int32_t* __restrict__ slot_ids) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int32_t s = ids[i];
    if (s >= 0) ids[i] = slot_ids[s];
  }
}

static int lin_grid_ev(size_t n, int sm_count) {
  size_t g = (n + 255) / 256;
  if (g > (size_t)sm_count * 8) g = (size_t)sm_count * 8;
  return g < 1 ? 1 : (int)g;
}

}  // namespace fr

static void free_tracked(fr_ctx* h, void* p) {
  if (!p) return;
  for (auto& q : h->allocs) if (q == p) q = nullptr;
  cudaFree(p);
}

static int eval_ws_ensure(fr_ctx* h, size_t N, cudaStream_t st) {
  auto& e = h->ev;
  int rc;
  if (!e.owner_counts && (rc = dalloc(h, &e.owner_counts, 8))) return rc;
  if (N <= e.n_cap) return FR_OK;
  if (e.n_cap) {
    FR_CUDA(h, cudaStreamSynchronize(st));          // the old buffers may still be read by queued work
    for (void* p : {(void*)e.keys, (void*)e.flags, (void*)e.excl, (void*)e.scan_tmp, (void*)e.sort.k[0], (void*)e.sort.k[1],
                    (void*)e.sort.v[0], (void*)e.sort.v[1], (void*)e.sort.tile_hist, (void*)e.sort.ticket, (void*)e.sort.scan_tmp})
      free_tracked(h, p);
    e.sort = SortBufs{};
    e.n_cap = 0;
  }
  if ((rc = dalloc(h, &e.keys, N)) || (rc = dalloc(h, &e.flags, N)) || (rc = dalloc(h, &e.excl, N)) ||
      (rc = dalloc(h, &e.scan_tmp, N / 4096 + 2)) || (rc = alloc_sort(h, e.sort, N)))
    return rc;
  e.n_cap = N;
  return FR_OK;
}

extern "C" int fr_shard_eval_plan(fr_handle h, const int32_t* cand, const int32_t* n_cand, int32_t n_users,
                                  int32_t cand_stride, int32_t world, int32_t num_items_global, int32_t cap,
                                  int32_t* req, int32_t* slots, int32_t* slot_ids, float* cand_cats_out, float* out_flag,
                                  fr_stream s) {
  if (!h || !h->has_tables) return fail(h, FR_ERR_STATE, "fr_set_tables first");
  if (n_users < 0 || cand_stride <= 0 || cand_stride > 128 || world < 1 || world > 8 || cap < 1 || num_items_global < 1)
    return fail(h, FR_ERR_ARG, "fr_shard_eval_plan: need n_users >= 0, 0 < cand_stride <= 128, 1 <= world <= 8, cap >= 1, "
                "num_items_global >= 1");
  const int64_t ipr = ((int64_t)num_items_global + world - 1) / world;
  if (ipr != h->cfg.num_items)
    return fail(h, FR_ERR_ARG, "fr_shard_eval_plan: ceil(%d / %d) != local Recipe_Embedding rows %d", num_items_global, world,
                h->cfg.num_items);
  if ((int64_t)world * cap > INT32_MAX) return fail(h, FR_ERR_ARG, "world * cap exceeds int32");
  if (!req || !slot_ids || !out_flag || (n_users > 0 && (!cand || !n_cand || !slots)))
    return fail(h, FR_ERR_ARG, "null pointer");
  if (cand_cats_out && !h->tab.item_cats) return fail(h, FR_ERR_ARG, "cand_cats_out needs the global item_cats table");
  const size_t N = (size_t)n_users * cand_stride;
  if (N >= (size_t)1 << 31) return fail(h, FR_ERR_ARG, "n_users * cand_stride exceeds 2^31 (evaluate in rounds)");
  cudaStream_t st = (cudaStream_t)s;
  const size_t n_slots = (size_t)world * cap;
  FR_CUDA(h, cudaMemsetAsync(req, 0xff, n_slots * sizeof(int32_t), st));
  FR_CUDA(h, cudaMemsetAsync(slot_ids, 0xff, n_slots * sizeof(int32_t), st));
  if (N == 0) return FR_OK;                     // a rank without test users requests nothing (and still serves)
  int rc = eval_ws_ensure(h, N, st); if (rc) return rc;
  auto& e = h->ev;
  FR_CUDA(h, cudaMemsetAsync(e.owner_counts, 0, 8 * sizeof(uint32_t), st));
  EvalPlanParams p{};
  p.cand = cand; p.n_cand = n_cand; p.N = (uint32_t)N; p.stride = cand_stride; p.W = world;
  p.ipr = (uint32_t)ipr; p.n_items = (uint32_t)num_items_global; p.cap = (uint32_t)cap;
  p.item_cats = (const float4*)h->tab.item_cats; p.cats_out = (float4*)cand_cats_out;
  p.keys = e.keys; p.flags = e.flags; p.excl = e.excl; p.owner_counts = e.owner_counts;
  p.req = req; p.slots = slots; p.slot_ids = slot_ids; p.flag = out_flag;
  const int grid = lin_grid_ev(N, h->sm_count);
  eval_plan_keys_kernel<<<grid, 256, 0, st>>>(p); ++g_launches;
  const int r = radix_sort_pairs(e.sort, e.keys, (uint32_t)N, nullptr, bits_for((int64_t)world * ipr + 1), st, h->sm_count);
  p.keys_sorted = e.sort.k[r]; p.perm = e.sort.v[r];
  eval_plan_heads_kernel<<<grid, 256, 0, st>>>(p); ++g_launches;
  exclusive_scan_u32(e.flags, e.excl, (uint32_t)N, e.scan_tmp, nullptr, st);
  eval_plan_fill_kernel<<<grid, 256, 0, st>>>(p); ++g_launches;
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}

extern "C" int fr_shard_eval_serve(fr_handle h, const int32_t* rreq, int32_t n, void* rows, fr_stream s) {
  if (!h || !h->has_tables) return fail(h, FR_ERR_STATE, "fr_set_tables first");
  if (n < 0 || (n > 0 && (!rreq || !rows))) return fail(h, FR_ERR_ARG, "null argument");
  if (n == 0) return FR_OK;
  cudaStream_t st = (cudaStream_t)s;
  int rc = shadow_sync(h, st); if (rc) return rc;
  Launch l{h->sm_count, st, nullptr};
  PeerPtrs none{}; none.world = 0;
  launch_gather_rows((const float4*)h->tab.R, rreq, (uint32_t)n, h->mc.DV, (float4*)rows, none, l, (uint32_t)h->cfg.num_items,
                     h->table_bf16 ? 2 : 0);
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}

extern "C" int fr_eval_sampled_rows(fr_handle h, const int32_t* users, int32_t user_rows, const int32_t* slots,
                                    const int32_t* n_cand, int32_t n_users, int32_t cand_stride, const float* cand_cats, const void* rows,
                                    int32_t n_rows, const int32_t* slot_ids, int32_t K, int32_t* topk_ids, int32_t* gt_rank,
                                    float* scores, fr_stream s) {
  if (!h || !h->has_tables) return fail(h, FR_ERR_STATE, "fr_set_tables first");
  if (n_users < 0 || cand_stride <= 0 || cand_stride > 128 || K <= 0 || n_rows < 1 || user_rows < 0 ||
      user_rows > h->cfg.num_users)
    return fail(h, FR_ERR_ARG, "need 0<cand_stride<=128, K>0, n_rows>=1, 0<=user_rows<=Personal_Memory rows");
  if (n_users > 0 && (!users || !slots || !n_cand || !cand_cats || !rows || !slot_ids || !topk_ids || !gt_rank))
    return fail(h, FR_ERR_ARG, "null pointer (cand_cats is required: the slots do not index item_cats)");
  if ((int64_t)n_rows * h->mc.DV >= (1ll << 32))
    return fail(h, FR_ERR_UNSUPPORTED, "fr_eval_sampled_rows: %d rows of %d exceed 2^32 16-byte groups", n_rows, h->mc.D);
  if (n_users == 0) return FR_OK;
  cudaStream_t st = (cudaStream_t)s;
  { int rc = shadow_sync(h, st); if (rc) return rc; }
  Launch l{h->sm_count, st, nullptr};
  // a user row at or past user_rows (the padding of the last user shard) is outside Personal_Memory: empty rank list
  launch_eval_sampled(h->mc, (const float4*)h->tab.P, (const float4*)rows, (const float4*)h->tab.Cat, users, slots, n_cand,
                      n_users, cand_stride, (const float4*)cand_cats, nullptr, K, topk_ids, gt_rank, scores, health_of(h), l,
                      user_rows, n_rows, h->table_bf16 ? 1 : 0);
  const size_t nk = (size_t)n_users * K;
  eval_unslot_kernel<<<lin_grid_ev(nk, h->sm_count), 256, 0, st>>>(topk_ids, nk, slot_ids); ++g_launches;
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}
