// Full-catalog top-K: index build (recipes grouped by category mask, bf16 B operand), per-pass
// user operand, exact fp64 re-ranking of the GEMM filter's survivors, exact fallback, cross-shard
// merge, and the fr_catalog_* C ABI.  The tcgen05 kernel itself is in catalog_gemm.cu; the maths
// and the error bound are stated in catalog.cuh.
#include <math_constants.h>

#include <algorithm>
#include <array>
#include <cstdlib>
#include <vector>

#include "catalog.cuh"
#include "ctx.h"

namespace fr {

#ifdef FR_CAT_TILE_BOUND
#define FR_CAT_M2R(w) , (w).margin2r
#else
#define FR_CAT_M2R(w)
#endif

struct CatalogWs {
  bool prepared = false;
  int cta_group = 1, epi_sets = 1, BN = 128, a_split = 0, I = 0, KP = 0, k_blocks = 0, n_tiles = 0, present = 0, n_valid_items = 0;
  int max_pass_rows = 0, force_splits = 0;
  // index (built by fr_catalog_prepare)
  uint32_t* keys = nullptr; SortBufs sortM; int32_t* gs_dev = nullptr;
  __nv_bfloat16* Bq = nullptr; int32_t *row_item = nullptr, *tile_group = nullptr, *tile_valid = nullptr, *tile_pos = nullptr;
  float* rmax = nullptr;
#ifdef FR_CAT_TILE_BOUND
  float *tile_rn = nullptr, *tile_rho = nullptr, *margin2r = nullptr;    // staged per-tile bound (catalog.cuh)
#endif
  const float4* item_cats = nullptr;      // [I,4] masks of THIS table's recipes (tables.item_cats unless overridden)
  int tiles_cap = 0;
  CUtensorMap tmB;
  // per-pass workspace
  int mp_cap = 0;
  __nv_bfloat16* A = nullptr; float *bias = nullptr, *margin2 = nullptr, *cand_sc = nullptr;
  int32_t *cand_row = nullptr, *cand_cnt = nullptr, *ovf = nullptr, *ovf_list = nullptr, *ovf_count = nullptr, *keff = nullptr;
  int32_t* call_ovf = nullptr;            // rows of the current call (all passes) that took the exact fallback
  double* scratch = nullptr; int exact_blocks = 0;
  unsigned long long* dbg = nullptr;
  uint32_t* ukeys = nullptr; SortBufs sortU; int32_t* block_first = nullptr;   // users sorted by best mask group
  int group_lo[16] = {0}, group_hi[16] = {0}, group_last_valid[16] = {0};
  // timing
  std::vector<std::array<cudaEvent_t, 5>> evs; size_t ev_used = 0;
  double t_sum[4] = {0, 0, 0, 0}; int64_t t_passes = 0;
};

// ------------------------------------------------------------------ index build
__global__ void cat_mask_kernel(const float4* __restrict__ item_cats, int I, uint32_t* __restrict__ keys) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= I) return;
  const float4 m = __ldg(item_cats + i);
  keys[i] = (m.x != 0.f ? 1u : 0u) | (m.y != 0.f ? 2u : 0u) | (m.z != 0.f ? 4u : 0u) | (m.w != 0.f ? 8u : 0u);
}

__global__ void cat_group_bounds_kernel(const uint32_t* __restrict__ sorted_keys, int I, int32_t* __restrict__ gs) {
  const uint32_t g = threadIdx.x;     // 0..16: first sorted position with key >= g
  if (g > 16) return;
  int lo = 0, hi = I;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (sorted_keys[mid] < g) lo = mid + 1; else hi = mid; }
  gs[g] = lo;
}

// one warp per padded row: B[row] = bf16(R[item]) (zero rows pad a group's last tile)
__global__ void __launch_bounds__(FR_THREADS)
cat_pack_items_kernel(const float4* __restrict__ R, int DV, int KP, const uint32_t* __restrict__ sorted_idx,
                      const int32_t* __restrict__ tile_valid, const int32_t* __restrict__ tile_pos, int n_rows, int BN,
                      __nv_bfloat16* __restrict__ Bq, int32_t* __restrict__ row_item, float* __restrict__ rmax
#ifdef FR_CAT_TILE_BOUND
                      , float* __restrict__ tile_rn
#endif
                      ) {
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * FR_WARPS_PER_BLOCK + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  const int tile = r / BN, j = r % BN;
  const bool valid = j < __ldg(tile_valid + tile);
  const int item = valid ? (int)__ldg(sorted_idx + __ldg(tile_pos + tile) + j) : -1;
  if (lane == 0) row_item[r] = item;
  float nrm = 0.f;
  uint2* dst = reinterpret_cast<uint2*>(Bq + (size_t)r * KP);
  for (int i = lane; i < KP / 4; i += 32) {
    float4 v = f4zero();
    if (valid && i < DV) v = __ldg(R + (size_t)item * DV + i);
    nrm += dot4(v, v);
    const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 o;
    o.x = *reinterpret_cast<const uint32_t*>(&lo); o.y = *reinterpret_cast<const uint32_t*>(&hi);
    dst[i] = o;
  }
  nrm = warp_sum(nrm);
  if (lane == 0 && valid) atomicMax(reinterpret_cast<int*>(rmax), __float_as_int(sqrtf(nrm) * 1.000001f));
#ifdef FR_CAT_TILE_BOUND
  if (lane == 0 && valid) atomicMax(reinterpret_cast<int*>(tile_rn + tile), __float_as_int(sqrtf(nrm) * 1.000001f));
#endif
}

#ifdef FR_CAT_TILE_BOUND
// rho[t] = (largest recipe norm of tile t) / (largest of the catalog), rounded up and clamped to (0, 1]
__global__ void cat_tile_rho_kernel(const float* __restrict__ tile_rn, const float* __restrict__ rmax, int n_tiles,
                                    float* __restrict__ rho) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tiles) return;
  const float m = *rmax;
  rho[t] = m > 0.f ? fminf(1.0f, __fmul_ru(__fdiv_ru(tile_rn[t], m), 1.000001f)) : 1.0f;
}
#endif

// ------------------------------------------------------------------ per-pass user operand
struct UserSrc {
  const float4* P;        // table or dense query rows
  const int32_t* uidx;    // nullable: row -> user id
  int row0;               // first query row of this pass
  const uint32_t* perm;   // nullable: pass row -> query row of the pass (users sorted by best mask group)
  HealthBlend hb;         // G != nullptr: rows are scored with the health term (table queries only)
  uint32_t n_table;       // rows of Personal_Memory when uidx indexes it: an id outside the table reads row 0 (never OOB;
                          // host lists are range-checked by the Python layer, which raises like tf.gather)
};
__device__ __forceinline__ int query_row(const UserSrc& s, int j) {      // index into the caller's user list / outputs
  return s.row0 + (s.perm ? (int)__ldg(s.perm + j) : j);
}
__device__ __forceinline__ int user_of(const UserSrc& s, int j) {
  const int qr = query_row(s, j);
  if (!s.uidx) return qr;
  const int u = __ldg(s.uidx + qr);
  return (uint32_t)u < s.n_table ? u : 0;
}
__device__ __forceinline__ const float4* user_row(const UserSrc& s, int j, int DV) {
  return s.P + (size_t)user_of(s, j) * 5 * DV;
}

// Exclusion lists (catalog.cuh): CSR over query rows, ids in the OUTPUT id space (local row * id_mul + id_add).
// An id is compared, never dereferenced: one this table cannot return (another shard's, out of range, negative) -> -1.
struct ExclLists {
  const int32_t* off;     // [n_users+1] or nullptr (no lists)
  const int32_t* ids;     // [nnz]
  int id_mul, id_add, n_items;
};
__device__ __forceinline__ int excl_local(const ExclLists& x, int id) {
  const long long d = (long long)id - x.id_add;
  if (d < 0) return -1;
  const uint32_t u = (uint32_t)d, m = (uint32_t)x.id_mul;   // d < 2^32 (two int32s); 32-bit division stays inline
  const uint32_t q = u / m;
  return (u - q * m == 0 && q < (uint32_t)x.n_items) ? (int)q : -1;
}

// key of a query row = the mask group with the largest category term a/|g| * sum_{c in g} <P[u,0],Cat[c]>
template <int NV>
__global__ void __launch_bounds__(FR_THREADS)
cat_user_key_kernel(UserSrc src, int n_rows, const float4* __restrict__ Cat, int DV, int present, uint32_t* __restrict__ keys) {
  const int lane = threadIdx.x & 31;
  const int j = blockIdx.x * FR_WARPS_PER_BLOCK + (threadIdx.x >> 5);
  if (j >= n_rows) return;
  float4 pr5[5][NV];
#pragma unroll
  for (int s5 = 0; s5 < 5; ++s5) load_row_ro<NV>(pr5[s5], user_row(src, j, DV) + (size_t)s5 * DV, DV, lane);
  health_blend_rows<NV>(pr5, src.hb, user_of(src, j), DV, lane);
  float4 (&p0)[NV] = pr5[0];
  float h[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int i = lane + 32 * k;
      if (i < DV) acc += dot4(p0[k], __ldg(Cat + c * DV + i));
    }
    h[c] = warp_sum(acc);
  }
  float best = -__int_as_float(0x7f800000);
  int gb = 0;
  for (int g = 1; g < 16; ++g) {
    if (!((present >> g) & 1)) continue;
    float hs = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) if ((g >> c) & 1) hs += h[c];
    hs /= (float)__popc(g);
    if (hs > best) { best = hs; gb = g; }
  }
  if (lane == 0) keys[j] = (uint32_t)gb;
}

template <int NV>
__global__ void __launch_bounds__(FR_THREADS)
cat_pack_users_kernel(UserSrc src, int n_rows, int m_pad, const float4* __restrict__ Cat, int DV, int KP, int a_split, float a,
                      float oma, int present, const float* __restrict__ rmax_p, float cfac,
                      __nv_bfloat16* __restrict__ A, float* __restrict__ bias, float* __restrict__ margin2,
                      int32_t* __restrict__ block_first, int block_rows, ExclLists excl, int K,
                      int32_t* __restrict__ keff, int32_t* __restrict__ ovf
#ifdef FR_CAT_TILE_BOUND
                      , float* __restrict__ margin2r
#endif
                      ) {
  const int lane = threadIdx.x & 31;
  const int j = blockIdx.x * FR_WARPS_PER_BLOCK + (threadIdx.x >> 5);
  if (j >= m_pad) return;
  const bool valid = j < n_rows;
  // K_eff of the row (in pass order, after the user sort): K + the listed ids that map into this table.  A row
  // whose K_eff exceeds CAT_MAXK is flagged to the exact fallback here (this also clears ovf for the pass).
  int ke = K;
  if (valid && excl.off) {
    const int qr = query_row(src, j);
    const int e0 = __ldg(excl.off + qr), e1 = __ldg(excl.off + qr + 1);
    int c = 0;
    for (int e = e0 + lane; e < e1; e += 32) c += excl_local(excl, __ldg(excl.ids + e)) >= 0 ? 1 : 0;
    ke += __reduce_add_sync(FR_FULL, c);
  }
  if (lane == 0) { keff[j] = min(ke, CAT_MAXK); ovf[j] = ke > CAT_MAXK ? 1 : 0; }
  float4 pr[5][NV];
  double h[4] = {0, 0, 0, 0};
  if (valid) {
    const float4* prow = user_row(src, j, DV);
#pragma unroll
    for (int s = 0; s < 5; ++s) load_row_ro<NV>(pr[s], prow + (size_t)s * DV, DV, lane);
    health_blend_rows<NV>(pr, src.hb, user_of(src, j), DV, lane);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      double acc = 0.0;
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        const int i = lane + 32 * k;
        if (i < DV) {
          const float4 cv = __ldg(Cat + c * DV + i);
          acc += (double)pr[0][k].x * cv.x + (double)pr[0][k].y * cv.y + (double)pr[0][k].z * cv.z + (double)pr[0][k].w * cv.w;
        }
      }
      h[c] = warp_sum_d(acc);
    }
  } else {
#pragma unroll
    for (int s = 0; s < 5; ++s)
#pragma unroll
      for (int k = 0; k < NV; ++k) pr[s][k] = f4zero();
  }
  const float rmax = __ldg(rmax_p);
  float emax = 0.f, bbest = -__int_as_float(0x7f800000);
#ifdef FR_CAT_TILE_BOUND
  float eround = 0.f;
#endif
  int gbest = 0;
  for (int g = 1; g < 16; ++g) {
    if (!((present >> g) & 1)) continue;
    const float inv_n = 1.0f / (float)__popc(g);
    float nrm = 0.f;
    const int KA = a_split ? 2 * KP : KP;       // row = [bf16 head | bf16 tail of the remainder]
    uint2* dst = reinterpret_cast<uint2*>(A + ((size_t)g * m_pad + j) * KA);
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int i = lane + 32 * k;
      if (i < KP / 4) {
        float4 z = f4zero();
        if (i < DV) {
#pragma unroll
          for (int c = 0; c < 4; ++c) if ((g >> c) & 1) z = add4(z, pr[1 + c][k]);
          z = scale4(oma * inv_n, z);
        }
        nrm += dot4(z, z);
        const __nv_bfloat162 lo = __floats2bfloat162_rn(z.x, z.y), hi = __floats2bfloat162_rn(z.z, z.w);
        uint2 o;
        o.x = *reinterpret_cast<const uint32_t*>(&lo); o.y = *reinterpret_cast<const uint32_t*>(&hi);
        dst[i] = o;
        if (a_split) {
          const float2 f0 = __bfloat1622float2(lo), f1 = __bfloat1622float2(hi);
          const __nv_bfloat162 t0 = __floats2bfloat162_rn(z.x - f0.x, z.y - f0.y), t1 = __floats2bfloat162_rn(z.z - f1.x, z.w - f1.y);
          uint2 o2;
          o2.x = *reinterpret_cast<const uint32_t*>(&t0); o2.y = *reinterpret_cast<const uint32_t*>(&t1);
          dst[KP / 4 + i] = o2;
        }
      }
    }
    nrm = warp_sum(nrm);
    double hs = 0.0;
#pragma unroll
    for (int c = 0; c < 4; ++c) if ((g >> c) & 1) hs += h[c];
    const float b = (float)((double)a * (hs / (double)__popc(g)));
    const float ar = sqrtf(nrm) * rmax;
#ifdef FR_CAT_TILE_BOUND
    emax = fmaxf(emax, cfac * ar);                                    // scales with the tile's largest recipe norm
    eround = fmaxf(eround, 4.76837158e-7f * (fabsf(b) + ar));         // 2^-21: the fp32 roundings of bias, bias - E, v + bias
#else
    const float E = cfac * ar + 4.76837158e-7f * (fabsf(b) + ar);     // 2^-21: fp32 rounding of bias and of v + bias
    emax = fmaxf(emax, E);
#endif
    if (b > bbest) { bbest = b; gbest = g; }
    if (lane == 0) bias[(size_t)g * m_pad + j] = b;
  }
  if (lane == 0) {
    margin2[j] = 2.0f * emax * 1.00001f;
#ifdef FR_CAT_TILE_BOUND
    margin2r[j] = 2.0f * eround * 1.00001f;
#endif
    if (block_first && j % block_rows == 0) block_first[j / block_rows] = gbest;   // the block sweeps this group first
  }
}

// ------------------------------------------------------------------ exact scoring + ranking helpers
// inference (Model_Recommender.py:56-97) for one (user, recipe) in fp64 from the fp32 tables.
// sP = the user's [5,D] row, sH[c] = <P[u,0], Cat[c]>.  All lanes return the score.
__device__ __forceinline__ double exact_score_warp(const float* sP, const double* sH, const float* __restrict__ Rrow,
                                                   const float4 m, int D, int lane, double a, double oma) {
  const bool m0 = m.x != 0.f, m1 = m.y != 0.f, m2 = m.z != 0.f, m3 = m.w != 0.f;
  const int n = (int)m0 + (int)m1 + (int)m2 + (int)m3;
  double acc = 0.0;
  for (int d = lane; d < D; d += 32) {
    double z = 0.0;
    if (m0) z += (double)sP[D + d];
    if (m1) z += (double)sP[2 * D + d];
    if (m2) z += (double)sP[3 * D + d];
    if (m3) z += (double)sP[4 * D + d];
    acc = fma(z, (double)__ldg(Rrow + d), acc);
  }
  acc = warp_sum_d(acc);
  double hs = 0.0;
  if (m0) hs += sH[0];
  if (m1) hs += sH[1];
  if (m2) hs += sH[2];
  if (m3) hs += sH[3];
  if (n == 0) return -CUDART_INF;
  return a * (hs / n) + oma * (acc / n);
}

__device__ __forceinline__ void load_user_exact(const UserSrc& src, int row, const float* __restrict__ Cat, int D, float* sP,
                                                double* sH, int tid, int nthreads) {
  const float* pf = reinterpret_cast<const float*>(user_row(src, row, D / 4));
  for (int i = tid; i < 5 * D; i += nthreads) sP[i] = __ldg(pf + i);
  __syncthreads();
  if (src.hb.G) { health_blend_flat(sP, src.hb, user_of(src, row), D, tid, nthreads); __syncthreads(); }
  const int warp = tid >> 5, lane = tid & 31;
  if (warp < 4) {
    double acc = 0.0;
    for (int d = lane; d < D; d += 32) acc = fma((double)sP[d], (double)__ldg(Cat + warp * D + d), acc);
    acc = warp_sum_d(acc);
    if (lane == 0) sH[warp] = acc;
  }
  __syncthreads();
}

__device__ __forceinline__ bool ranks_before(double sa, int ia, double sb, int ib) {
  return sa > sb || (sa == sb && ia < ib);      // score desc, id asc
}
__device__ void bitonic_rank_sort(double* s, int* id, int n2, int tid, int nthreads) {
  for (int k = 2; k <= n2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < n2; i += nthreads) {
        const int x = i ^ j;
        if (x > i) {
          const bool first = ranks_before(s[i], id[i], s[x], id[x]);
          const bool up = (i & k) == 0;
          if (up ? (!first && ranks_before(s[x], id[x], s[i], id[i])) : first) {
            const double ts = s[i]; s[i] = s[x]; s[x] = ts;
            const int ti = id[i]; id[i] = id[x]; id[x] = ti;
          }
        }
      }
      __syncthreads();
    }
  }
}

struct FinParams {
  UserSrc src;
  const float* R; const float* Cat; const float4* item_cats; const int32_t* row_item;
  int D, n_rows, m_pad, n_split, K;
  double a, oma;
  const float* margin2; const float* cand_sc; const int32_t* cand_row; const int32_t* cand_cnt;
#ifdef FR_CAT_TILE_BOUND
  const float* margin2r; const float* tile_rho; int bn_shift;
#endif
  const int32_t* ovf; int32_t* ovf_list; int32_t* ovf_count;   // ovf_count: this pass's fallback rows (the fallback's work list)
  int32_t* call_ovf;                        // the call's fallback rows over all passes (fr_catalog_fallback_rows)
  const int32_t* keff;                      // [m_pad] per-row K_eff
  ExclLists excl;                           // carries id_mul / id_add of the outputs too
  int id_mul, id_add;
  int32_t* out_ids; double* out_scores;     // [n_users, K]
};

constexpr int FIN_THREADS = 128;

__global__ void __launch_bounds__(FIN_THREADS) cat_finalize_kernel(const FinParams f) {
  extern __shared__ __align__(16) uint8_t fsm[];
  double* es = reinterpret_cast<double*>(fsm);                 // [FCAP]
  double* sH = es + CAT_FCAP;                                  // [4]
  int* eid = reinterpret_cast<int*>(sH + 4);                   // [FCAP]
  int* frow = eid + CAT_FCAP;                                  // [FCAP]
  float* sP = reinterpret_cast<float*>(frow + CAT_FCAP);       // [5*D]
  float* csc = sP + 5 * f.D;                                   // [n_split*CAP]
  int* crow = reinterpret_cast<int*>(csc + f.n_split * CAT_CAP);
  __shared__ int s_red[FIN_THREADS / 32];
  __shared__ int s_nF;
  __shared__ uint32_t s_hist[256], s_sel[2];
  const int row = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  bool overflow = f.ovf[row] != 0;
  int n_tot = 0;
  const int Ke = f.keff[row];
  if (!overflow) {
    for (int sp = 0; sp < f.n_split; ++sp) {
      const size_t lr = (size_t)sp * f.m_pad + row;
      const int c = f.cand_cnt[lr];
      for (int e = tid; e < c; e += FIN_THREADS) {
        csc[n_tot + e] = __ldcg(f.cand_sc + lr * CAT_CAP + e);
        crow[n_tot + e] = __ldcg(f.cand_row + lr * CAT_CAP + e);
      }
      n_tot += c;
    }
    if (tid == 0) s_nF = 0;
    __syncthreads();
    // tau = K_eff-th largest approximate score over the union of the split lists
    float lo = -__int_as_float(0x7f800000);
    if (n_tot > Ke) {
      // exact K-th largest key by 8-bit radix select over a shared-memory histogram: 4 passes x 3 barriers (the
      // bit-by-bit search it replaces cost 64 barriers and 32 sweeps over the list: 18 % of this kernel's instructions)
      uint32_t res = 0; uint32_t need = (uint32_t)Ke;
      for (int pass = 3; pass >= 0; --pass) {
        for (int b = tid; b < 256; b += FIN_THREADS) s_hist[b] = 0u;
        __syncthreads();
        const int sh = 8 * pass;
        for (int e = tid; e < n_tot; e += FIN_THREADS) {
          const uint32_t k = fkey(csc[e]);
          if (pass == 3 || (k >> (sh + 8)) == (res >> (sh + 8))) atomicAdd(&s_hist[(k >> sh) & 255u], 1u);
        }
        __syncthreads();
        if (warp == 0) {                       // lane l owns bins [8l, 8l+8); counts are taken from the top bin down
          uint32_t loc[8], sum = 0;
#pragma unroll
          for (int q = 0; q < 8; ++q) { loc[q] = s_hist[8 * lane + q]; sum += loc[q]; }
          uint32_t incl = sum;                 // sum over lanes >= this one
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_down_sync(FR_FULL, incl, o);
            if (lane + o < 32) incl += y;
          }
          uint32_t a = incl - sum;             // entries in higher bins than this lane's
          if (a < need && need <= incl) {
#pragma unroll
            for (int q = 7; q >= 0; --q) {
              if (a + loc[q] >= need) { s_sel[0] = (uint32_t)(8 * lane + q); s_sel[1] = need - a; break; }
              a += loc[q];
            }
          }
        }
        __syncthreads();
        res |= s_sel[0] << sh;
        need = s_sel[1];
      }
#ifdef FR_CAT_TILE_BOUND
      lo = funkey(res);                 // K_eff-th largest LOWER bound over the union of the lists
#else
      lo = __fsub_rd(funkey(res), f.margin2[row]);
#endif
    }
    for (int e = tid; e < n_tot; e += FIN_THREADS) {
#ifdef FR_CAT_TILE_BOUND
      if (__fadd_ru(__fmaf_ru(f.margin2[row], __ldg(f.tile_rho + (crow[e] >> f.bn_shift)), csc[e]), f.margin2r[row]) >= lo) {
#else
      if (csc[e] >= lo) {
#endif
        const int pos = atomicAdd(&s_nF, 1);
        if (pos < CAT_FCAP) frow[pos] = crow[e];
      }
    }
    __syncthreads();
    if (s_nF > CAT_FCAP) overflow = true;
  }
  // The row's listed recipes of this table (local ids; at most K_eff - K <= CAT_MAXK - 1 of them here) are staged in
  // the candidate area, free once the survivors are picked: s_ex[0] = count, s_ex[1..].  (No static shared memory is
  // added: one more KB would cost this kernel a resident block per SM.)
  int* s_ex = reinterpret_cast<int*>(csc);
  if (!overflow && f.excl.off) {
    if (tid == 0) s_ex[0] = 0;
    __syncthreads();
    const int qr = query_row(f.src, row);
    const int e1 = __ldg(f.excl.off + qr + 1);
    for (int e = __ldg(f.excl.off + qr) + tid; e < e1; e += FIN_THREADS) {
      const int l = excl_local(f.excl, __ldg(f.excl.ids + e));
      if (l >= 0) { const int pos = atomicAdd(s_ex, 1); if (pos < CAT_MAXK) s_ex[1 + pos] = l; }
    }
  }
  if (overflow) {                       // exact fallback takes this row
    if (tid == 0) { const int slot = atomicAdd(f.ovf_count, 1); f.ovf_list[slot] = row; atomicAdd(f.call_ovf, 1); }
    return;
  }
  const int nF = s_nF;
  load_user_exact(f.src, row, f.Cat, f.D, sP, sH, tid, FIN_THREADS);
  // Re-score, ONE THREAD PER SURVIVOR.  (A warp per survivor made this stage a chain of dependent
  // L2/HBM reads -- id, mask, row -- per survivor: 35 % of a cfg2 run.)  Ids and masks of all survivors
  // are fetched first; the fp64 user row sum_{c in g} P[u,1+c] is built once per mask that occurs; then
  // every thread streams its survivor's recipe row with independent 16-byte loads.
  double* Z = reinterpret_cast<double*>(crow + f.n_split * CAT_CAP);      // [16][D], after the candidate arrays
  __shared__ int s_masks;
  if (tid == 0) s_masks = 0;
  __syncthreads();
  const int nex = f.excl.off ? min(s_ex[0], CAT_MAXK) : 0;
  for (int i = tid; i < nF; i += FIN_THREADS) {
    const int item = __ldg(f.row_item + frow[i]);
    const float4 m = __ldg(f.item_cats + item);
    int g = (m.x != 0.f ? 1 : 0) | (m.y != 0.f ? 2 : 0) | (m.z != 0.f ? 4 : 0) | (m.w != 0.f ? 8 : 0);
    for (int x = 0; x < nex; ++x)               // a listed survivor is scored like a recipe without a category: -inf
      if (s_ex[1 + x] == item) { g = 0; break; }
    eid[i] = item;
    frow[i] = g;                                   // the padded row is no longer needed: keep the mask
    atomicOr(&s_masks, 1 << g);
  }
  __syncthreads();
  const int present = s_masks;
  for (int e = tid; e < 16 * f.D; e += FIN_THREADS) {
    const int g = e / f.D, d = e % f.D;
    if ((present >> g) & 1) {
      double z = 0.0;
      if (g & 1) z += (double)sP[f.D + d];
      if (g & 2) z += (double)sP[2 * f.D + d];
      if (g & 4) z += (double)sP[3 * f.D + d];
      if (g & 8) z += (double)sP[4 * f.D + d];
      Z[e] = z;
    }
  }
  __syncthreads();
  for (int i = tid; i < nF; i += FIN_THREADS) {
    const int g = frow[i], n = __popc(g);
    const float4* rr = reinterpret_cast<const float4*>(f.R + (size_t)eid[i] * f.D);
    const double* zg = Z + g * f.D;
    double acc = 0.0;
#pragma unroll 8
    for (int q = 0; q < f.D / 4; ++q) {
      const float4 r = __ldg(rr + q);
      acc = fma(zg[4 * q], (double)r.x, acc);
      acc = fma(zg[4 * q + 1], (double)r.y, acc);
      acc = fma(zg[4 * q + 2], (double)r.z, acc);
      acc = fma(zg[4 * q + 3], (double)r.w, acc);
    }
    double hs = 0.0;
    if (g & 1) hs += sH[0];
    if (g & 2) hs += sH[1];
    if (g & 4) hs += sH[2];
    if (g & 8) hs += sH[3];
    es[i] = n ? f.a * (hs / n) + f.oma * (acc / n) : -CUDART_INF;
  }
  __syncthreads();
  // Final order by counting: the rank of a survivor is the number of survivors that come before it in
  // (score desc, id asc) -- a strict total order, ids are distinct.  nF is a few hundred: nF^2/128 broadcast
  // shared loads per thread and no barrier, against ~40 barrier-separated bitonic stages.
  const size_t ob = (size_t)query_row(f.src, row) * f.K;
  int n_real = 0;
  for (int i = tid; i < nF; i += FIN_THREADS) {
    const double si = es[i];
    const int ii = eid[i];
    if (si > -CUDART_INF) {
      int rank = 0;
      for (int j = 0; j < nF; ++j) rank += ranks_before(es[j], eid[j], si, ii) ? 1 : 0;
      if (rank < f.K) {
        f.out_ids[ob + rank] = ii * f.id_mul + f.id_add;
        if (f.out_scores) f.out_scores[ob + rank] = si;
      }
    }
  }
  for (int i = tid; i < nF; i += FIN_THREADS) n_real += es[i] > -CUDART_INF ? 1 : 0;
  n_real = __reduce_add_sync(FR_FULL, n_real);
  if (lane == 0) s_red[warp] = n_real;
  __syncthreads();
  n_real = s_red[0] + s_red[1] + s_red[2] + s_red[3];
  for (int k = n_real + tid; k < f.K; k += FIN_THREADS) {        // fewer recipes than K: pad
    f.out_ids[ob + k] = -1;
    if (f.out_scores) f.out_scores[ob + k] = -CUDART_INF;
  }
}

// ------------------------------------------------------------------ exact fallback (rows the filter gave up on)
__device__ __forceinline__ unsigned long long dkey(double d) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(d);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ULL);
}

constexpr int EX_THREADS = 1024;

// Phase A of the parallel fallback: exact scores of EVERY recipe for up to gridDim.y fallback rows
// [slot0, slot0 + gridDim.y), spread over the whole GPU (blockIdx.x = recipe slice).
constexpr int EXS_THREADS = 256, EXS_ITEMS = 4096;
__global__ void __launch_bounds__(EXS_THREADS) cat_exact_scores_kernel(const FinParams f, int I, int slot0,
                                                                      double* __restrict__ scratch) {
  __shared__ float sP[5 * 256];
  __shared__ double sH[4];
  const int slot = slot0 + blockIdx.y;
  if (slot >= min(*f.ovf_count, f.m_pad)) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  load_user_exact(f.src, f.ovf_list[slot], f.Cat, f.D, sP, sH, tid, EXS_THREADS);
  double* sc = scratch + (size_t)blockIdx.y * I;
  const int i0 = blockIdx.x * EXS_ITEMS, i1 = min(I, i0 + EXS_ITEMS);
  for (int item = i0 + warp; item < i1; item += EXS_THREADS / 32) {
    const double s = exact_score_warp(sP, sH, f.R + (size_t)item * f.D, __ldg(f.item_cats + item), f.D, lane, f.a, f.oma);
    if (lane == 0) sc[item] = s;
  }
}

// Phase B (scores_ready: one block per row of the round, scores in scratch[blockIdx.x]) or the
// self-contained tail (one block scores and selects row after row: complete but slow).
__global__ void __launch_bounds__(EX_THREADS) cat_exact_kernel(const FinParams f, int I, double* __restrict__ scratch,
                                                               int slot0, int scores_ready) {
  __shared__ float sP[5 * 256];
  __shared__ double sH[4];
  __shared__ unsigned hist[256];
  __shared__ unsigned long long s_prefix;
  __shared__ int s_need, s_ngt, wcnt[EX_THREADS / 32];
  __shared__ double ss[CAT_MAXK];
  __shared__ int sid[CAT_MAXK];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double* sc = scratch + (size_t)blockIdx.x * I;
  const int n_ov = min(*f.ovf_count, f.m_pad);
  const int Keff = min(f.K, I);
  for (int slot = slot0 + blockIdx.x; slot < n_ov; slot += scores_ready ? (1 << 30) : gridDim.x) {
    const int row = f.ovf_list[slot];
    __syncthreads();
    if (!scores_ready) {
      load_user_exact(f.src, row, f.Cat, f.D, sP, sH, tid, EX_THREADS);
      for (int item = warp; item < I; item += EX_THREADS / 32) {
        const double s = exact_score_warp(sP, sH, f.R + (size_t)item * f.D, __ldg(f.item_cats + item), f.D, lane, f.a, f.oma);
        if (lane == 0) sc[item] = s;
      }
    }
    __syncthreads();
    if (f.excl.off) {                           // listed recipes leave the ranking (-inf is padded with -1 below)
      const int qr = query_row(f.src, row);
      const int e1 = __ldg(f.excl.off + qr + 1);
      for (int e = __ldg(f.excl.off + qr) + tid; e < e1; e += EX_THREADS) {
        const int l = excl_local(f.excl, __ldg(f.excl.ids + e));
        if (l >= 0) sc[l] = -CUDART_INF;
      }
      __syncthreads();
    }
    // radix select of the Keff-th largest 64-bit key
    unsigned long long prefix = 0;
    int need = Keff;
    for (int pass = 7; pass >= 0; --pass) {
      for (int b = tid; b < 256; b += EX_THREADS) hist[b] = 0;
      __syncthreads();
      for (int i = tid; i < I; i += EX_THREADS) {
        const unsigned long long k = dkey(sc[i]);
        if (pass == 7 || (k >> (8 * (pass + 1))) == prefix) atomicAdd(&hist[(k >> (8 * pass)) & 255ULL], 1u);
      }
      __syncthreads();
      if (tid == 0) {
        int acc = 0, b = 255;
        for (; b > 0; --b) { if (acc + (int)hist[b] >= need) break; acc += (int)hist[b]; }
        s_prefix = (prefix << 8) | (unsigned long long)b;
        s_need = need - acc;
      }
      __syncthreads();
      prefix = s_prefix; need = s_need;
      __syncthreads();
    }
    const unsigned long long kth = prefix;      // `need` recipes with key == kth complete the top-K: lowest ids first
    if (tid == 0) s_ngt = 0;
    __syncthreads();
    for (int i = tid; i < I; i += EX_THREADS)
      if (dkey(sc[i]) > kth) { const int pos = atomicAdd(&s_ngt, 1); if (pos < CAT_MAXK) { ss[pos] = sc[i]; sid[pos] = i; } }
    __syncthreads();
    const int ngt = s_ngt;
    int base = 0;
    for (int start = 0; start < I && base < need; start += EX_THREADS) {
      const int i = start + tid;
      const bool flag = i < I && dkey(sc[i]) == kth;
      const uint32_t bal = __ballot_sync(FR_FULL, flag);
      if (lane == 0) wcnt[warp] = __popc(bal);
      __syncthreads();
      int wp = 0, total = 0;
      for (int w = 0; w < EX_THREADS / 32; ++w) { const int c = wcnt[w]; if (w < warp) wp += c; total += c; }
      const int pos = base + wp + __popc(bal & ((1u << lane) - 1u));
      if (flag && pos < need && ngt + pos < CAT_MAXK) { ss[ngt + pos] = sc[i]; sid[ngt + pos] = i; }
      base += total;
      __syncthreads();
    }
    int n2 = 2;
    while (n2 < Keff) n2 <<= 1;
    for (int i = Keff + tid; i < n2; i += EX_THREADS) { ss[i] = -CUDART_INF; sid[i] = 0x7fffffff; }
    __syncthreads();
    bitonic_rank_sort(ss, sid, n2, tid, EX_THREADS);
    const size_t ob = (size_t)query_row(f.src, row) * f.K;
    for (int k = tid; k < f.K; k += EX_THREADS) {
      const bool has = k < Keff && ss[k] > -CUDART_INF;
      f.out_ids[ob + k] = has ? sid[k] * f.id_mul + f.id_add : -1;
      if (f.out_scores) f.out_scores[ob + k] = has ? ss[k] : -CUDART_INF;
    }
  }
}

// ------------------------------------------------------------------ cross-shard merge
__global__ void __launch_bounds__(FIN_THREADS)
cat_merge_kernel(const int32_t* __restrict__ ids, const double* __restrict__ scores, int n_lists, int n_users, int K,
                 int32_t* __restrict__ out_ids, double* __restrict__ out_scores) {
  extern __shared__ __align__(16) uint8_t msm[];
  const int n = n_lists * K;
  int n2 = 2;
  while (n2 < n) n2 <<= 1;
  double* s = reinterpret_cast<double*>(msm);
  int* id = reinterpret_cast<int*>(s + n2);
  const int u = blockIdx.x, tid = threadIdx.x;
  for (int e = tid; e < n2; e += FIN_THREADS) {
    double sv = -CUDART_INF; int iv = 0x7fffffff;
    if (e < n) {
      const int l = e / K, k = e % K;
      const size_t src = ((size_t)l * n_users + u) * K + k;
      const int i0 = ids[src];
      if (i0 >= 0) { iv = i0; sv = scores[src]; }
    }
    s[e] = sv; id[e] = iv;
  }
  __syncthreads();
  bitonic_rank_sort(s, id, n2, tid, FIN_THREADS);
  for (int k = tid; k < K; k += FIN_THREADS) {
    const bool has = id[k] != 0x7fffffff;
    out_ids[(size_t)u * K + k] = has ? id[k] : -1;
    if (out_scores) out_scores[(size_t)u * K + k] = has ? s[k] : -CUDART_INF;
  }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// bf16 row-major [rows, KP] -> boxes of [box_rows, 64] with the 128-byte swizzle
static int make_tmap(fr_ctx* h, CUtensorMap* m, void* base, uint64_t rows, int KP, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(h, FR_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
  const cuuint64_t gdim[2] = {(cuuint64_t)KP, rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)KP * 2};
  const cuuint32_t box[2] = {(cuuint32_t)CAT_BK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, gdim, gstride, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(h, FR_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return FR_OK;
}

}  // namespace fr

void catalog_free(fr_ctx* h) {
  if (!h || !h->cat) return;
  for (auto& s : h->cat->evs) for (auto& e : s) cudaEventDestroy(e);
  delete h->cat;
  h->cat = nullptr;
}

extern "C" int fr_catalog_prepare(fr_handle h, const fr_catalog_opts* opts, const float* item_cats, fr_stream s) {
  if (!h) return FR_ERR_ARG;
  if (!h->has_tables) return fail(h, FR_ERR_STATE, "fr_set_tables first");
  if (!item_cats) item_cats = h->tab.item_cats;
  if (!item_cats) return fail(h, FR_ERR_STATE, "catalog scoring needs the recipes' category masks (dish_to_category)");
  if ((uintptr_t)item_cats & 15) return fail(h, FR_ERR_ARG, "item_cats must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(s);
  cudaDeviceProp prop;
  FR_CUDA(h, cudaGetDeviceProperties(&prop, h->device));
  if (prop.major != 10) return fail(h, FR_ERR_UNSUPPORTED, "catalog scoring is tcgen05 code: needs sm_100, device is sm_%d%d", prop.major, prop.minor);
  if (!h->cat) h->cat = new CatalogWs();
  CatalogWs& w = *h->cat;
  w.item_cats = reinterpret_cast<const float4*>(item_cats);
  const int I = h->cfg.num_items, D = h->mc.D, DV = h->mc.DV;
  const int KP = (D + CAT_BK - 1) / CAT_BK * CAT_BK;
  int rc;
  if (w.I != I) {
    if (w.I != 0) return fail(h, FR_ERR_STATE, "catalog index was built for %d recipes", w.I);
    w.I = I; w.KP = KP; w.k_blocks = KP / CAT_BK;
    w.tiles_cap = (I + 16 * CAT_BN_MAX) / 128 + 1;   // every mask group pads its last tile: <= 15 * 255 extra rows; sized in narrow tiles
    if ((rc = dalloc(h, &w.keys, (size_t)I))) return rc;
    if ((rc = alloc_sort(h, w.sortM, (size_t)I))) return rc;
    if ((rc = dalloc(h, &w.gs_dev, 17))) return rc;
    if ((rc = dalloc(h, &w.Bq, (size_t)w.tiles_cap * 128 * KP))) return rc;
    if ((rc = dalloc(h, &w.row_item, (size_t)w.tiles_cap * 128))) return rc;
    if ((rc = dalloc(h, &w.tile_group, (size_t)w.tiles_cap))) return rc;
    if ((rc = dalloc(h, &w.tile_valid, (size_t)w.tiles_cap))) return rc;
    if ((rc = dalloc(h, &w.tile_pos, (size_t)w.tiles_cap))) return rc;
    if ((rc = dalloc(h, &w.rmax, 1))) return rc;
#ifdef FR_CAT_TILE_BOUND
    if ((rc = dalloc(h, &w.tile_rn, (size_t)w.tiles_cap))) return rc;
    if ((rc = dalloc(h, &w.tile_rho, (size_t)w.tiles_cap))) return rc;
#endif
    FR_CUDA(h, catalog_gemm_configure());
    FR_CUDA(h, cudaFuncSetAttribute(cat_finalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  }
  w.cta_group = (opts && opts->cta_group == 1) ? 1 : 2;
  w.BN = (opts && opts->tile_n == 128) ? 128 : 256;
  w.a_split = (w.k_blocks * 2 <= CAT_KB_MAX && !(opts && opts->a_split == 1)) ? 1 : 0;   // opts->a_split: 0 default (on when it fits), 1 off
  const int BN = w.BN;
  w.max_pass_rows = (opts && opts->max_pass_rows > 0) ? opts->max_pass_rows : 0;
  w.epi_sets = (opts && (opts->epi_sets == 1 || opts->epi_sets == 2 || opts->epi_sets == 4)) ? opts->epi_sets : 1;
  w.force_splits = (opts && opts->splits > 0) ? std::min(opts->splits, CAT_LISTS_MAX / w.epi_sets) : 0;

  cat_mask_kernel<<<(I + 255) / 256, 256, 0, st>>>(w.item_cats, I, w.keys);
  ++g_launches;
  FR_CHECK_LAUNCH(h);
  const int r = radix_sort_pairs(w.sortM, w.keys, (uint32_t)I, nullptr, 4, st, h->sm_count);
  cat_group_bounds_kernel<<<1, 32, 0, st>>>(w.sortM.k[r], I, w.gs_dev);
  ++g_launches;
  FR_CHECK_LAUNCH(h);
  int32_t gs[17];
  FR_CUDA(h, cudaMemcpyAsync(gs, w.gs_dev, sizeof(gs), cudaMemcpyDeviceToHost, st));
  FR_CUDA(h, cudaStreamSynchronize(st));
  std::vector<int32_t> tg, tv, tp;
  w.present = 0;
  for (int g = 1; g < 16; ++g) {
    const int cnt = gs[g + 1] - gs[g];
    if (cnt <= 0) continue;
    w.present |= 1 << g;
    for (int o = 0; o < cnt; o += BN) { tg.push_back(g); tv.push_back(std::min(BN, cnt - o)); tp.push_back(gs[g] + o); }
  }
  for (int g = 0; g < 16; ++g) w.group_lo[g] = w.group_hi[g] = 0;
  for (int t = 0; t < (int)tg.size(); ++t) {
    if (w.group_hi[tg[t]] == 0) w.group_lo[tg[t]] = t;
    w.group_hi[tg[t]] = t + 1;
    w.group_last_valid[tg[t]] = tv[t];
  }
  w.n_tiles = (int)tg.size();
  w.n_valid_items = I - (gs[1] - gs[0]);
  if (w.n_tiles > w.tiles_cap) return fail(h, FR_ERR_STATE, "catalog tile count %d exceeds capacity %d", w.n_tiles, w.tiles_cap);
  if (w.n_tiles > 0) {
    FR_CUDA(h, cudaMemcpyAsync(w.tile_group, tg.data(), tg.size() * 4, cudaMemcpyHostToDevice, st));
    FR_CUDA(h, cudaMemcpyAsync(w.tile_valid, tv.data(), tv.size() * 4, cudaMemcpyHostToDevice, st));
    FR_CUDA(h, cudaMemcpyAsync(w.tile_pos, tp.data(), tp.size() * 4, cudaMemcpyHostToDevice, st));
    FR_CUDA(h, cudaMemsetAsync(w.rmax, 0, 4, st));
#ifdef FR_CAT_TILE_BOUND
    FR_CUDA(h, cudaMemsetAsync(w.tile_rn, 0, (size_t)w.n_tiles * 4, st));
#endif
    const int n_rows = w.n_tiles * BN;
    cat_pack_items_kernel<<<(n_rows + FR_WARPS_PER_BLOCK - 1) / FR_WARPS_PER_BLOCK, FR_THREADS, 0, st>>>(
        reinterpret_cast<const float4*>(h->tab.R), DV, KP, w.sortM.v[r], w.tile_valid, w.tile_pos, n_rows, BN, w.Bq,
        w.row_item, w.rmax
#ifdef FR_CAT_TILE_BOUND
        , w.tile_rn
#endif
        );
    ++g_launches;
#ifdef FR_CAT_TILE_BOUND
    cat_tile_rho_kernel<<<(w.n_tiles + 255) / 256, 256, 0, st>>>(w.tile_rn, w.rmax, w.n_tiles, w.tile_rho);
    ++g_launches;
#endif
    FR_CHECK_LAUNCH(h);
    FR_CUDA(h, cudaStreamSynchronize(st));     // host vectors above go out of scope
    if ((rc = make_tmap(h, &w.tmB, w.Bq, (uint64_t)w.n_tiles * BN, KP, BN / w.cta_group))) return rc;
  }
  w.prepared = true;
  return FR_OK;
}

// (Re)allocation of a pass buffer: the buffer it had is freed first (cudaFree waits for the device).
static void pass_free(fr_ctx* h, void* p) {
  if (p) for (auto& q : h->allocs) if (q == p) { cudaFree(q); q = nullptr; }
}
template <class T>
static int pass_alloc(fr_ctx* h, T** p, size_t n) {
  pass_free(h, *p);
  *p = nullptr;
  return dalloc(h, p, n);
}

// Pass workspace for passes of up to mp rows.  A later call that needs more rows than it has (a re-prepare with a
// larger max_pass_rows, or the defaults after a small one) replaces the row-sized buffers once the stream is idle.
static int catalog_ensure_pass_ws(fr_ctx* h, CatalogWs& w, int mp, cudaStream_t st) {
  if (mp <= w.mp_cap) return FR_OK;
  if (w.mp_cap != 0) FR_CUDA(h, cudaStreamSynchronize(st));
  w.mp_cap = 0;                     // until every buffer below has its new size
  int rc;
  const size_t R = (size_t)mp;
  if ((rc = pass_alloc(h, &w.A, 16 * R * w.KP * 2))) return rc;
  if ((rc = pass_alloc(h, &w.bias, 16 * R))) return rc;
  if ((rc = pass_alloc(h, &w.margin2, R))) return rc;
#ifdef FR_CAT_TILE_BOUND
  if ((rc = pass_alloc(h, &w.margin2r, R))) return rc;
#endif
  const size_t RL = R * 4;          // candidate lists: up to 4 column sets per (split, row)
  if ((rc = pass_alloc(h, &w.cand_sc, RL * CAT_CAP))) return rc;
  if ((rc = pass_alloc(h, &w.cand_row, RL * CAT_CAP))) return rc;
  if ((rc = pass_alloc(h, &w.cand_cnt, RL))) return rc;
  if ((rc = pass_alloc(h, &w.ovf, R))) return rc;
  if ((rc = pass_alloc(h, &w.keff, R))) return rc;
  if ((rc = pass_alloc(h, &w.ovf_list, R))) return rc;
  if ((rc = pass_alloc(h, &w.ukeys, R))) return rc;
  for (void* p : {(void*)w.sortU.k[0], (void*)w.sortU.k[1], (void*)w.sortU.v[0], (void*)w.sortU.v[1], (void*)w.sortU.tile_hist,
                  (void*)w.sortU.ticket, (void*)w.sortU.scan_tmp})
    pass_free(h, p);
  w.sortU = SortBufs();
  if ((rc = alloc_sort(h, w.sortU, R))) return rc;
  if ((rc = pass_alloc(h, &w.block_first, R / CAT_BM + 1))) return rc;
  if (!w.scratch) {                 // sized by the catalog, not by the pass
    if ((rc = dalloc(h, &w.ovf_count, 1))) return rc;
    if ((rc = dalloc(h, &w.call_ovf, 1))) return rc;
    if ((rc = dalloc(h, &w.dbg, 8))) return rc;
    FR_CUDA(h, cudaMemset(w.dbg, 0, 64));
    const size_t budget = (size_t)512 << 20;
    w.exact_blocks = (int)std::max<size_t>(2, std::min<size_t>((size_t)h->sm_count, budget / ((size_t)w.I * 8)));
    if ((rc = dalloc(h, &w.scratch, (size_t)w.exact_blocks * w.I))) return rc;
  }
  w.mp_cap = mp;
  return FR_OK;
}

extern "C" int fr_catalog_topk_excluding(fr_handle h, const int32_t* users, const float* P_rows, int32_t n_users, int32_t K,
                                         const int32_t* excl_off, const int32_t* excl_ids, int32_t id_mul, int32_t id_add,
                                         int32_t* out_ids, double* out_scores, fr_stream s) {
  if (!h || !out_ids || n_users < 0) return FR_ERR_ARG;
  if (!h->cat || !h->cat->prepared) return fail(h, FR_ERR_STATE, "fr_catalog_prepare first");
  if (K <= 0 || K > CAT_MAXK) return fail(h, FR_ERR_UNSUPPORTED, "K must be in [1,%d], got %d", CAT_MAXK, K);
  if ((excl_off == nullptr) != (excl_ids == nullptr))
    return fail(h, FR_ERR_ARG, "excl_off and excl_ids are given together (both NULL: no lists)");
  if (excl_off && id_mul < 1) return fail(h, FR_ERR_ARG, "id_mul must be >= 1 with exclusion lists, got %d", id_mul);
  if (n_users == 0) return FR_OK;
  if (P_rows && h->health_blend) return fail(h, FR_ERR_ARG, "the health term needs user ids (labels): pass users, not dense P_rows");
  if (h->table_bf16) return fail(h, FR_ERR_UNSUPPORTED, "fr_catalog_* reads fp32 tables (exact fp64 re-rank): not available with bf16 tables");
  if (!P_rows) { const int rcs = shadow_sync(h, static_cast<cudaStream_t>(s)); if (rcs) return rcs; }
  if (!P_rows && !users && n_users > h->cfg.num_users)
    return fail(h, FR_ERR_ARG, "n_users=%d exceeds the %d rows of Personal_Memory", n_users, h->cfg.num_users);
  CatalogWs& w = *h->cat;
  cudaStream_t st = static_cast<cudaStream_t>(s);
  const int CG = w.cta_group, BMC = CAT_BM * CG;
  const int n_clusters = std::max(1, h->sm_count / CG);
  // rows per pass: whole waves of user blocks; small calls split the recipe sweep instead
  const int pass_rows = w.max_pass_rows > 0 ? (w.max_pass_rows + BMC - 1) / BMC * BMC : n_clusters * BMC * 4;
  const int NSET = w.epi_sets;
  int rc = catalog_ensure_pass_ws(h, w, std::max(pass_rows, 2 * n_clusters * BMC), st);
  if (rc) return rc;
  FR_CUDA(h, cudaMemsetAsync(w.call_ovf, 0, 4, st));
  const int D = h->mc.D, DV = h->mc.DV;
  // |s_hat - s| <= cfac * |A||R|.  bf16 rounding u = 2^-8 on both operands: 2u + u^2; with the split
  // user operand (exact to 2^-16) only the recipe side rounds: u + 2^-15.  Plus fp32 accumulation.
  const float cfac = (w.a_split ? 0.00390625f + 3.1e-5f : 0.0078278f) + (float)w.KP * (w.a_split ? 2.f : 1.f) * 9.54e-7f;
  const bool timing = h->timing;

  for (int row0 = 0; row0 < n_users; row0 += pass_rows) {
    const int rows = std::min(pass_rows, n_users - row0);
    const int m_blocks = (rows + BMC - 1) / BMC, m_pad = m_blocks * BMC;
    int n_split = w.force_splits ? w.force_splits : (n_clusters + m_blocks - 1) / m_blocks;
    n_split = std::max(1, std::min({n_split, CAT_LISTS_MAX / NSET, std::max(1, w.n_tiles)}));
    while (n_split > 1 && (size_t)n_split * m_pad > (size_t)w.mp_cap) --n_split;
    const int n_lists = n_split * NSET;
    const int tps = std::max(1, (w.n_tiles + n_split - 1) / n_split);
    UserSrc src{reinterpret_cast<const float4*>(P_rows ? P_rows : h->tab.P), P_rows ? nullptr : users, row0, nullptr, health_of(h),
                (uint32_t)h->cfg.num_users};
    const ExclLists excl{excl_off, excl_ids, id_mul, id_add, w.I};

    std::array<cudaEvent_t, 5>* ev = nullptr;
    if (timing) {
      if (w.ev_used == w.evs.size()) {
        w.evs.emplace_back();
        for (auto& e : w.evs.back()) FR_CUDA(h, cudaEventCreate(&e));
      }
      ev = &w.evs[w.ev_used++];
      FR_CUDA(h, cudaEventRecord((*ev)[0], st));
    }
    const float4* Cat4 = reinterpret_cast<const float4*>(h->tab.Cat);
    const bool sorted = n_split == 1 && w.n_tiles > 0;      // whole sweeps: sort users by best mask group
    if (sorted) {
      const int kgrid = (rows + FR_WARPS_PER_BLOCK - 1) / FR_WARPS_PER_BLOCK;
      if (h->NV == 1) cat_user_key_kernel<1><<<kgrid, FR_THREADS, 0, st>>>(src, rows, Cat4, DV, w.present, w.ukeys);
      else cat_user_key_kernel<2><<<kgrid, FR_THREADS, 0, st>>>(src, rows, Cat4, DV, w.present, w.ukeys);
      ++g_launches;
      FR_CHECK_LAUNCH(h);
      const int r = radix_sort_pairs(w.sortU, w.ukeys, (uint32_t)rows, nullptr, 4, st, h->sm_count);
      src.perm = w.sortU.v[r];
    }
    int32_t* bf = sorted ? w.block_first : nullptr;
    const int pgrid = (m_pad + FR_WARPS_PER_BLOCK - 1) / FR_WARPS_PER_BLOCK;
    if (h->NV == 1)
      cat_pack_users_kernel<1><<<pgrid, FR_THREADS, 0, st>>>(src, rows, m_pad, Cat4, DV, w.KP, w.a_split, h->mc.a, h->mc.oma, w.present,
                                                            w.rmax, cfac, w.A, w.bias, w.margin2, bf, BMC, excl, K, w.keff, w.ovf
                                                            FR_CAT_M2R(w));
    else
      cat_pack_users_kernel<2><<<pgrid, FR_THREADS, 0, st>>>(src, rows, m_pad, Cat4, DV, w.KP, w.a_split, h->mc.a, h->mc.oma, w.present,
                                                            w.rmax, cfac, w.A, w.bias, w.margin2, bf, BMC, excl, K, w.keff, w.ovf
                                                            FR_CAT_M2R(w));
    ++g_launches;
    FR_CHECK_LAUNCH(h);
    FR_CUDA(h, cudaMemsetAsync(w.cand_cnt, 0, (size_t)n_lists * m_pad * 4, st));
    FR_CUDA(h, cudaMemsetAsync(w.ovf_count, 0, 4, st));
    if (ev) FR_CUDA(h, cudaEventRecord((*ev)[1], st));

    if (w.n_tiles > 0) {
      CUtensorMap tmA;
      if ((rc = make_tmap(h, &tmA, w.A, (uint64_t)16 * m_pad, w.a_split ? 2 * w.KP : w.KP, CAT_BM))) return rc;
      CatGemmParams p{};
      p.m_blocks = m_blocks; p.m_pad = m_pad; p.n_rows = rows; p.n_split = n_split; p.tiles_per_split = tps;
      p.n_tiles = w.n_tiles; p.k_blocks = w.k_blocks; p.keff = w.keff; p.a_split = w.a_split;
      // diagnostics / tuning switches (environment; never needed for results): FOODREC_CATALOG_DEBUG = ceiling
      // measurements (catalog.cuh), _DENSE_MIN / _BOOT_TILES = epilogue regime knobs, _CYCLES = in-kernel cycle counters
      { const char* dm = getenv("FOODREC_CATALOG_DEBUG"); p.debug_mode = dm ? atoi(dm) : 0; }
      p.tile_group = w.tile_group; p.tile_valid = w.tile_valid; p.bias = w.bias; p.margin2 = w.margin2;
#ifdef FR_CAT_TILE_BOUND
      p.tile_rho = w.tile_rho; p.margin2r = w.margin2r; p.bn_shift = w.BN == 256 ? 8 : 7;
#endif
      p.block_first = bf;
      { const char* dmn = getenv("FOODREC_CATALOG_DENSE_MIN"); p.dense_min = dmn ? atoi(dmn) : 3; }
      {   // bootstrap length: as many tiles as chunk maxima fit one candidate list (64 tiles = 16k recipes by default)
        const int chunks_per_tile = (w.BN / NSET) / 32;
        const char* bt = getenv("FOODREC_CATALOG_BOOT_TILES");
        p.boot_tiles = bt ? atoi(bt) : CAT_CAP / chunks_per_tile;
        p.boot_tiles = std::max(0, std::min(p.boot_tiles, CAT_CAP / chunks_per_tile));
      }
      p.dbg = getenv("FOODREC_CATALOG_CYCLES") ? w.dbg : nullptr;
      for (int g = 0; g < 16; ++g) { p.group_lo[g] = w.group_lo[g]; p.group_hi[g] = w.group_hi[g]; p.group_last_valid[g] = w.group_last_valid[g]; }
      p.cand_sc = w.cand_sc; p.cand_row = w.cand_row; p.cand_cnt = w.cand_cnt; p.ovf = w.ovf;
      launch_catalog_gemm(CG, NSET, w.BN, h->sm_count, tmA, w.tmB, p, st);
      FR_CHECK_LAUNCH(h);
    }
    if (ev) FR_CUDA(h, cudaEventRecord((*ev)[2], st));

    FinParams f{};
    f.src = src; f.R = h->tab.R; f.Cat = h->tab.Cat; f.item_cats = w.item_cats;
    f.row_item = w.row_item; f.D = D; f.n_rows = rows; f.m_pad = m_pad; f.n_split = n_lists; f.K = K;
    f.a = (double)h->mc.a; f.oma = (double)h->mc.oma;
    f.margin2 = w.margin2; f.cand_sc = w.cand_sc; f.cand_row = w.cand_row; f.cand_cnt = w.cand_cnt;
#ifdef FR_CAT_TILE_BOUND
    f.margin2r = w.margin2r; f.tile_rho = w.tile_rho; f.bn_shift = w.BN == 256 ? 8 : 7;
#endif
    f.ovf = w.ovf; f.ovf_list = w.ovf_list; f.ovf_count = w.ovf_count; f.call_ovf = w.call_ovf; f.keff = w.keff; f.excl = excl;
    f.id_mul = id_mul; f.id_add = id_add; f.out_ids = out_ids; f.out_scores = out_scores;
    const size_t fsm = (size_t)CAT_FCAP * (8 + 4 + 4) + 32 + (size_t)5 * D * 4 + (size_t)n_lists * CAT_CAP * 8 +
                       (size_t)16 * D * 8 + 8;      // + the per-mask fp64 user rows of the re-rank
    cat_finalize_kernel<<<rows, FIN_THREADS, fsm, st>>>(f);
    ++g_launches;
    FR_CHECK_LAUNCH(h);
    if (ev) FR_CUDA(h, cudaEventRecord((*ev)[3], st));
    // Rows the filter gave up on (massive ties): a few rounds of whole-GPU exact scoring + one-block
    // selection per row, then a self-contained tail for anything beyond (blocks exit at once when
    // there is nothing to do -- the common case).
    constexpr int EX_ROUNDS = 4;
    const int xs = (w.I + EXS_ITEMS - 1) / EXS_ITEMS;
    for (int r = 0; r < EX_ROUNDS; ++r) {
      cat_exact_scores_kernel<<<dim3(xs, w.exact_blocks), EXS_THREADS, 0, st>>>(f, w.I, r * w.exact_blocks, w.scratch);
      cat_exact_kernel<<<w.exact_blocks, EX_THREADS, 0, st>>>(f, w.I, w.scratch, r * w.exact_blocks, 1);
      g_launches += 2;
    }
    cat_exact_kernel<<<w.exact_blocks, EX_THREADS, 0, st>>>(f, w.I, w.scratch, EX_ROUNDS * w.exact_blocks, 0);
    ++g_launches;
    FR_CHECK_LAUNCH(h);
    if (ev) FR_CUDA(h, cudaEventRecord((*ev)[4], st));
  }
  return FR_OK;
}

extern "C" int fr_catalog_topk(fr_handle h, const int32_t* users, const float* P_rows, int32_t n_users, int32_t K,
                               int32_t id_mul, int32_t id_add, int32_t* out_ids, double* out_scores, fr_stream s) {
  return fr_catalog_topk_excluding(h, users, P_rows, n_users, K, nullptr, nullptr, id_mul, id_add, out_ids, out_scores, s);
}

extern "C" int fr_catalog_merge(fr_handle h, const int32_t* ids, const double* scores, int32_t n_lists,
                                int32_t n_users, int32_t K, int32_t* out_ids, double* out_scores, fr_stream s) {
  if (!h || !ids || !scores || !out_ids || n_lists <= 0 || n_users < 0 || K <= 0) return FR_ERR_ARG;
  if ((int64_t)n_lists * K > 4096) return fail(h, FR_ERR_UNSUPPORTED, "n_lists*K must be <= 4096");
  if (n_users == 0) return FR_OK;
  int n2 = 2;
  while (n2 < n_lists * K) n2 <<= 1;
  static bool configured = false;
  if (!configured) {
    FR_CUDA(h, cudaFuncSetAttribute(cat_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 4096 * 12));
    configured = true;
  }
  cat_merge_kernel<<<n_users, FIN_THREADS, (size_t)n2 * 12, static_cast<cudaStream_t>(s)>>>(ids, scores, n_lists, n_users, K,
                                                                                         out_ids, out_scores);
  ++g_launches;
  FR_CHECK_LAUNCH(h);
  return FR_OK;
}

extern "C" int fr_catalog_timing_read(fr_handle h, double* ms_sum, int64_t* n_passes, int32_t reset) {
  if (!h || !ms_sum) return FR_ERR_ARG;
  if (!h->cat) return fail(h, FR_ERR_STATE, "fr_catalog_prepare first");
  CatalogWs& w = *h->cat;
  for (size_t i = 0; i < w.ev_used; ++i) {
    auto& ev = w.evs[i];
    cudaEventSynchronize(ev[4]);
    for (int k = 0; k < 4; ++k) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, ev[k], ev[k + 1]) == cudaSuccess) w.t_sum[k] += ms;
    }
    w.t_passes += 1;
  }
  w.ev_used = 0;
  for (int k = 0; k < 4; ++k) ms_sum[k] = w.t_sum[k];
  if (n_passes) *n_passes = w.t_passes;
  if (reset) { for (double& t : w.t_sum) t = 0; w.t_passes = 0; }
  return FR_OK;
}

extern "C" int fr_catalog_fallback_rows(fr_handle h, int32_t* out, fr_stream s) {
  if (!h || !out) return FR_ERR_ARG;
  if (!h->cat || !h->cat->call_ovf) return fail(h, FR_ERR_STATE, "no catalog pass has run");
  cudaStream_t st = static_cast<cudaStream_t>(s);
  FR_CUDA(h, cudaMemcpyAsync(out, h->cat->call_ovf, 4, cudaMemcpyDeviceToHost, st));
  FR_CUDA(h, cudaStreamSynchronize(st));
  return FR_OK;
}

extern "C" int fr_catalog_cycle_counters(fr_handle h, uint64_t* out /* [8] */, fr_stream s) {
  if (!h || !out) return FR_ERR_ARG;
  if (!h->cat || !h->cat->dbg) return fail(h, FR_ERR_STATE, "no catalog pass has run");
  cudaStream_t st = static_cast<cudaStream_t>(s);
  FR_CUDA(h, cudaMemcpyAsync(out, h->cat->dbg, 64, cudaMemcpyDeviceToHost, st));
  FR_CUDA(h, cudaMemsetAsync(h->cat->dbg, 0, 64, st));
  FR_CUDA(h, cudaStreamSynchronize(st));
  return FR_OK;
}

extern "C" int fr_catalog_info(fr_handle h, int32_t* out /* [8] */) {
  if (!h || !out) return FR_ERR_ARG;
  if (!h->cat || !h->cat->prepared) return fail(h, FR_ERR_STATE, "fr_catalog_prepare first");
  const CatalogWs& w = *h->cat;
  out[0] = w.cta_group + 10 * w.a_split; out[1] = w.KP; out[2] = w.n_tiles; out[3] = w.present; out[4] = w.n_valid_items;
  out[5] = w.epi_sets * 1000 + w.BN; out[6] = CAT_CAP; out[7] = w.exact_blocks;
  return FR_OK;
}
