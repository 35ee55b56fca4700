// Negative sampler for 1:N training and sampled evaluation (BASELINE configs[4]: 1:8 negatives).  The reference has no
// sampler (get_train_instances takes listed negatives, Train_recommender.py:86-93); this is the counter-based
// equivalent so that host and device draw the SAME negatives for the same (seed, sample index): Philox4x32-10 (Salmon
// et al., SC'11; the generator curand and torch use), one counter per (sample, negative, attempt), uniform over [0, I)
// by multiply-shift.
//   counter = (sample_lo, sample_hi, negative j, attempt), key = (seed_lo, seed_hi)
//   cand    = mulhi32(x0, I);  the first of 16 attempts with cand != anchor and cand not in H(u) is taken
//   else    the first c of (anchor+1) % I, (anchor+2) % I, ... with c != anchor and c not in H(u); none: (anchor+1) % I
// H(u) = the user's history (fr_set_user_history), empty unless the call asks for it: then the rule is the
// positive-only rejection this sampler always had, bit for bit.  oracle/sampler_oracle.py restates it in numpy; ids are
// compared bit for bit.
#include "common.cuh"
#include "ctx.h"

namespace fr {

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
    const uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += W0; k.y += W1;
  }
  return c;
}

// first index k of the ascending row with row[k] >= v
__device__ __forceinline__ int row_lower_bound(const int32_t* __restrict__ row, int len, int32_t v) {
  int lo = 0, hi = len;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(row + mid) < v) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// Step 2 of the rule: walk c = (p+1) % I, (p+2) % I, ... alongside the sorted row from the lower bound of the start,
// wrapping once.  c only advances past p or past a value of the row, so the walk takes at most |row| + 2 steps.
__device__ __noinline__ uint32_t cyclic_unseen(const int32_t* __restrict__ row, int len, uint32_t p, uint32_t I) {
  const uint32_t c0 = (p + 1u) % I;
  uint32_t c = c0;
  int k = row_lower_bound(row, len, (int32_t)c0);
  bool wrapped = false;
  for (;;) {
    if (c == I) {
      if (wrapped) break;
      wrapped = true; c = 0; k = 0;
    }
    if (wrapped && c == c0) break;                       // every recipe is p or in the history (step 3)
    if (c == p) { ++c; continue; }
    while (k < len && __ldg(row + k) < (int32_t)c) ++k;
    if (k < len && __ldg(row + k) == (int32_t)c) { ++c; continue; }
    return c;
  }
  return c0;
}

// THE rule (one copy for every layout).  HIST = false: no history, the code of the positive-only sampler.
template <bool HIST>
__device__ __forceinline__ uint32_t draw_negative(unsigned long long g, uint32_t j, uint32_t p, uint32_t I, uint2 key,
                                                  const int32_t* __restrict__ row, int len) {
  for (uint32_t attempt = 0; attempt < 16; ++attempt) {
    const uint4 x = philox4x32_10(make_uint4((uint32_t)g, (uint32_t)(g >> 32), j, attempt), key);
    const uint32_t cand = __umulhi(x.x, I);
    if (cand == p) continue;
    if (HIST) {
      const int k = row_lower_bound(row, len, (int32_t)cand);
      if (k < len && __ldg(row + k) == (int32_t)cand) continue;
    }
    return cand;
  }
  if (HIST) return cyclic_unseen(row, len, p, I);
  return (p + 1u) % I;
}

struct UserHistory {
  const int32_t* off;   // [rows+1]
  const int32_t* ids;
  int32_t rows;         // a user outside [0, rows) has an empty history
};

// One thread per (sample s, negative j); sample index g = offset + s.  Layouts (FR_SAMPLE_*):
//   NEG        out_items [n, n_neg]
//   BPR        out_users[t] = users[s], out_items[2t] = anchor, [2t+1] = negative  (t = s*n_neg + j; one 8-byte store)
//   POINTWISE  rows s*(1+n_neg) + (0 | 1+j): (user, anchor, 1) then (user, negative_j, 0)
//   CAND       out_items [n, 1+n_neg] = [anchor, negatives...]
template <bool HIST, int LAYOUT>
__global__ void __launch_bounds__(256)
sample_kernel(const int32_t* __restrict__ users, const int32_t* __restrict__ pos, long long n, int n_neg, uint32_t I,
              uint2 key, unsigned long long offset, UserHistory hist, int32_t* __restrict__ out_users,
              int32_t* __restrict__ out_items, float* __restrict__ out_labels) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * n_neg) return;
  const long long s = t / n_neg;
  const uint32_t j = (uint32_t)(t % n_neg);
  const unsigned long long g = offset + (unsigned long long)s;
  const uint32_t p = (uint32_t)pos[s];
  const int32_t* row = nullptr;
  int len = 0;
  if (HIST) {
    const int32_t u = users[s];
    if (u >= 0 && u < hist.rows) {
      const int32_t a = __ldg(hist.off + u);
      row = hist.ids + a; len = __ldg(hist.off + u + 1) - a;
    }
  }
  const uint32_t item = draw_negative<HIST>(g, j, p, I, key, row, len);
  if (LAYOUT == FR_SAMPLE_NEG) {
    out_items[t] = (int32_t)item;
  } else if (LAYOUT == FR_SAMPLE_BPR) {
    out_users[t] = users[s];
    reinterpret_cast<int2*>(out_items)[t] = make_int2((int32_t)p, (int32_t)item);
  } else if (LAYOUT == FR_SAMPLE_POINTWISE) {
    const long long r = s * (n_neg + 1);
    const int32_t u = users[s];
    if (j == 0) { out_users[r] = u; out_items[r] = (int32_t)p; out_labels[r] = 1.f; }
    out_users[r + 1 + j] = u; out_items[r + 1 + j] = (int32_t)item; out_labels[r + 1 + j] = 0.f;
  } else {
    const long long r = s * (n_neg + 1);
    if (j == 0) out_items[r] = (int32_t)p;
    out_items[r + 1 + j] = (int32_t)item;
  }
}

// one warp per row: flag bit 1 = off[0] != 0, 2 = a row with off[u+1] < off[u] (or a negative offset), 4 = a row that
// is not ascending.  A row's ids are read only when its offsets are sound.
__global__ void __launch_bounds__(256)
history_check_kernel(const int32_t* __restrict__ off, const int32_t* __restrict__ ids, int32_t rows, uint32_t* flag) {
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
  if (blockIdx.x == 0 && threadIdx.x == 0 && off[0] != 0) atomicOr(flag, 1u);
  for (long long u = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; u < rows; u += warps) {
    const int32_t a = off[u], b = off[u + 1];
    if (a < 0 || b < a) { if (lane == 0) atomicOr(flag, 2u); continue; }
    bool bad = false;
    for (long long k = (long long)a + lane; k + 1 < b; k += 32) bad |= ids[k] > ids[k + 1];
    if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(flag, 4u);
  }
}

// raw generator output, exported so the tests can pin it to the published known-answer vectors
__global__ void philox_kat_kernel(const uint32_t* __restrict__ in, int n, uint32_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint4 x = philox4x32_10(make_uint4(in[6 * i], in[6 * i + 1], in[6 * i + 2], in[6 * i + 3]),
                                make_uint2(in[6 * i + 4], in[6 * i + 5]));
  out[4 * i] = x.x; out[4 * i + 1] = x.y; out[4 * i + 2] = x.z; out[4 * i + 3] = x.w;
}

template <bool HIST>
static void launch_sample(int layout, unsigned blocks, cudaStream_t st, const int32_t* users, const int32_t* pos, long long n,
                          int n_neg, uint32_t I, uint2 key, unsigned long long offset, UserHistory hist, int32_t* out_users,
                          int32_t* out_items, float* out_labels) {
#define FR_SAMPLE_LAUNCH(L) sample_kernel<HIST, L><<<blocks, 256, 0, st>>>(users, pos, n, n_neg, I, key, offset, hist, \
                                                                           out_users, out_items, out_labels)
  switch (layout) {
    case FR_SAMPLE_NEG: FR_SAMPLE_LAUNCH(FR_SAMPLE_NEG); break;
    case FR_SAMPLE_BPR: FR_SAMPLE_LAUNCH(FR_SAMPLE_BPR); break;
    case FR_SAMPLE_POINTWISE: FR_SAMPLE_LAUNCH(FR_SAMPLE_POINTWISE); break;
    default: FR_SAMPLE_LAUNCH(FR_SAMPLE_CAND); break;
  }
#undef FR_SAMPLE_LAUNCH
}

}  // namespace fr

// arguments checked by the entry points
static int sample_launch(fr_handle h, int32_t layout, const int32_t* users, const int32_t* anchors, int64_t n, int32_t n_neg,
                         uint64_t seed, uint64_t sample_offset, int64_t num_items, bool use_history, int32_t* out_users,
                         int32_t* out_items, float* out_labels, fr_stream s) {
  if (n == 0) return FR_OK;
  const long long total = (long long)n * n_neg;
  const unsigned blocks = (unsigned)((total + 255) / 256);
  const cudaStream_t st = static_cast<cudaStream_t>(s);
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  const UserHistory hist{h->hist_off, h->hist_ids, h->cfg.num_users};
  if (use_history)
    launch_sample<true>(layout, blocks, st, users, anchors, (long long)n, n_neg, (uint32_t)num_items, key,
                        (unsigned long long)sample_offset, hist, out_users, out_items, out_labels);
  else
    launch_sample<false>(layout, blocks, st, users, anchors, (long long)n, n_neg, (uint32_t)num_items, key,
                         (unsigned long long)sample_offset, hist, out_users, out_items, out_labels);
  ++g_launches;
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}

extern "C" int fr_set_user_history(fr_handle h, const int32_t* off, const int32_t* ids, fr_stream s) {
  if (!h) return FR_ERR_ARG;
  h->hist_off = h->hist_ids = nullptr;
  if (!off && !ids) return FR_OK;
  if (!off || !ids) return fail(h, FR_ERR_ARG, "fr_set_user_history: give both off and ids (or both NULL to clear)");
  if (!h->hist_flag) { int rc = dalloc(h, &h->hist_flag, 1); if (rc) return rc; }
  const cudaStream_t st = static_cast<cudaStream_t>(s);
  const int32_t rows = h->cfg.num_users;
  FR_CUDA(h, cudaMemsetAsync(h->hist_flag, 0, sizeof(uint32_t), st));
  const long long need = ((long long)rows * 32 + 255) / 256;
  const unsigned blocks = (unsigned)std::max(1ll, std::min(need, (long long)h->sm_count * 16));
  history_check_kernel<<<blocks, 256, 0, st>>>(off, ids, rows, h->hist_flag);
  ++g_launches;
  FR_CHECK_LAUNCH(h);
  uint32_t flag = 0;
  FR_CUDA(h, cudaMemcpyAsync(&flag, h->hist_flag, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  FR_CUDA(h, cudaStreamSynchronize(st));
  if (flag & 1u) return fail(h, FR_ERR_ARG, "fr_set_user_history: off[0] must be 0");
  if (flag & 2u) return fail(h, FR_ERR_ARG, "fr_set_user_history: offsets must be non-decreasing");
  if (flag & 4u) return fail(h, FR_ERR_ARG, "fr_set_user_history: every row must be ascending (duplicates allowed)");
  h->hist_off = off; h->hist_ids = ids;
  return FR_OK;
}

extern "C" int fr_sample_batch(fr_handle h, int32_t layout, const int32_t* users, const int32_t* anchors, int64_t n,
                               int32_t n_neg, uint64_t seed, uint64_t sample_offset, int64_t num_items, int32_t use_history,
                               int32_t* out_users, int32_t* out_items, float* out_labels, fr_stream s) {
  if (!h) return FR_ERR_ARG;
  if (layout < FR_SAMPLE_NEG || layout > FR_SAMPLE_CAND) return fail(h, FR_ERR_ARG, "fr_sample_batch: unknown layout %d", layout);
  if (!anchors || !out_items || n < 0 || n_neg <= 0) return fail(h, FR_ERR_ARG, "fr_sample_batch: anchors, out_items, n >= 0, n_neg > 0");
  const bool with_users = layout == FR_SAMPLE_BPR || layout == FR_SAMPLE_POINTWISE;
  if ((with_users || use_history) && !users) return fail(h, FR_ERR_ARG, "fr_sample_batch: this layout / the history needs users");
  if (with_users && !out_users) return fail(h, FR_ERR_ARG, "fr_sample_batch: this layout needs out_users");
  if (layout == FR_SAMPLE_POINTWISE && !out_labels) return fail(h, FR_ERR_ARG, "fr_sample_batch: FR_SAMPLE_POINTWISE needs out_labels");
  if (num_items == 0) num_items = h->cfg.num_items;
  if (num_items < 2 || num_items > 0x7fffffffll) return fail(h, FR_ERR_ARG, "negative sampling needs 2 <= num_items < 2^31");
  if (layout == FR_SAMPLE_BPR && (reinterpret_cast<uintptr_t>(out_items) & 7) != 0)
    return fail(h, FR_ERR_ARG, "out_items must be 8-byte aligned");
  if (use_history && !h->hist_off) return fail(h, FR_ERR_STATE, "fr_sample_batch: use_history without a history (fr_set_user_history)");
  return sample_launch(h, layout, users, anchors, n, n_neg, seed, sample_offset, num_items, use_history != 0, out_users,
                       out_items, out_labels, s);
}

extern "C" int fr_sample_negatives(fr_handle h, const int32_t* pos_items, int64_t n, int32_t n_neg, uint64_t seed,
                                   uint64_t sample_offset, int32_t* out, fr_stream s) {
  if (!h || !pos_items || !out || n < 0 || n_neg <= 0) return FR_ERR_ARG;
  if (h->cfg.num_items < 2) return fail(h, FR_ERR_ARG, "negative sampling needs at least 2 recipes");
  return sample_launch(h, FR_SAMPLE_NEG, nullptr, pos_items, n, n_neg, seed, sample_offset, h->cfg.num_items, false, nullptr,
                       out, nullptr, s);
}

extern "C" int fr_sample_bpr_batch(fr_handle h, const int32_t* users, const int32_t* pos_items, int64_t n, int32_t n_neg,
                                   uint64_t seed, uint64_t sample_offset, int64_t num_items, int32_t* out_users,
                                   int32_t* out_items, fr_stream s) {
  if (!h || !users || !pos_items || !out_users || !out_items || n < 0 || n_neg <= 0) return FR_ERR_ARG;
  if (num_items == 0) num_items = h->cfg.num_items;
  if (num_items < 2 || num_items > 0x7fffffffll) return fail(h, FR_ERR_ARG, "negative sampling needs 2 <= num_items < 2^31");
  if ((reinterpret_cast<uintptr_t>(out_items) & 7) != 0) return fail(h, FR_ERR_ARG, "out_items must be 8-byte aligned");
  return sample_launch(h, FR_SAMPLE_BPR, users, pos_items, n, n_neg, seed, sample_offset, num_items, false, out_users,
                       out_items, nullptr, s);
}

extern "C" int fr_philox4x32_10(fr_handle h, const uint32_t* ctr_key /* [n,6] device */, int32_t n, uint32_t* out /* [n,4] */,
                                fr_stream s) {
  if (!h || !ctr_key || !out || n < 0) return FR_ERR_ARG;
  if (n == 0) return FR_OK;
  philox_kat_kernel<<<(n + 127) / 128, 128, 0, static_cast<cudaStream_t>(s)>>>(ctr_key, n, out);
  ++g_launches;
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}
