// Full-catalog top-K (extension of evaluate.py: inference :56-97 over EVERY recipe).
// Shared declarations of catalog.cu / catalog_gemm.cu.
//
// score(u,i) = a * sum_c w_ic <P[u,0],Cat[c]>  +  (1-a) * sum_c w_ic <P[u,1+c], R[i]>
//            =        bias[u, mask_i]          +  < A[mask_i][u] , R[i] >
// with mask_i the recipe's category set (<= 15 non-empty masks), w_ic = m_ic / n_i,
//   A[g][u] = (1-a)/|g| * sum_{c in g} P[u,1+c]        (one D-vector per (mask, user))
//   bias[g][u] = a/|g| * sum_{c in g} <P[u,0],Cat[c]>  (fp64 -> fp32)
// Recipes are grouped by mask (stable sort, so ids ascend inside a group) and padded to
// whole 256-row tiles; a tile therefore has ONE mask, the dense contraction is
// [users x D] x [D x recipes] in bf16 on tcgen05 with fp32 accumulators in TMEM, and the
// category term is a per-(row, tile) constant the epilogue folds into its threshold.
//
// The bf16 GEMM is a FILTER with a proven error bound, not the answer:
//   |s_hat - s| <= E[u,t] = cfac * |A[g][u]| * max_{i in tile t} |R[i]|  (+ fp32 rounding of the bias add)
// The candidate lists hold LOWER bounds s_hat - E[u,t]; tau_run = the K-th largest lower bound so far (monotone, never
// above the true K-th best score); the epilogue keeps every recipe whose UPPER bound s_hat + E[u,t] reaches tau_run,
// which provably contains the exact top-K (oracle/catalog_filter_model.py states and property-tests the rule).  The
// bound is PER TILE: one heavy recipe (a hot item after training) widens the margin of its own 256-recipe tile only.
// The survivors (K + a few dozen) are re-scored in fp64 from the fp32 tables and ranked by (score desc, id asc).  Rows
// whose candidate list overflows (massive ties) fall back to an exact full scan.
//
// Exclusion lists (fr_catalog_topk_excluding): a query row may list recipe ids it must not get back (the user's
// training positives).  The filter still runs over ALL recipes, with a per-row K_eff = K + (entries of the row's list
// that map into this table; duplicates counted, which only widens the filter): tau_eff = the K_eff-th largest lower
// bound.  At most K_eff - K of the K_eff largest lower bounds belong to listed recipes, so at least K UNLISTED recipes
// have true score >= lower bound >= tau_eff: the K-th best unlisted score is >= tau_eff >= tau_run at any time, and a
// member of the exact unlisted top-K has upper bound >= its score >= tau_run -- it is kept.  Listed survivors are then
// dropped where scores are exact (the fp64 re-rank, or -inf in the exact fallback's score row).  K_eff > CAT_MAXK:
// the row goes to the exact fallback up front.
#pragma once
// Per-tile filter bound (default).  -DFR_CAT_GLOBAL_BOUND builds the round-1 filter whose margin uses the largest
// recipe norm of the WHOLE catalog (kept for A/B runs: foodrec_b200._build.build_variant("globalbound", [...])).
#if !defined(FR_CAT_GLOBAL_BOUND) && !defined(FR_CAT_TILE_BOUND)
#define FR_CAT_TILE_BOUND 1
#endif
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace fr {

constexpr int CAT_BM = 128;        // user rows per CTA (TMEM lanes)
constexpr int CAT_BN_MAX = 256;    // recipes per tile: 256 (2 accumulator stages in TMEM) or 128 (4 stages)
constexpr int CAT_BK = 64;         // bf16 elements per 128-byte swizzle atom
constexpr int CAT_KB_MAX = 4;      // D <= 256
constexpr int CAT_CAP = 512;       // candidate slots per (split, user)
constexpr int CAT_FCAP = 512;      // survivors re-scored per user (more: exact fallback)
constexpr int CAT_MAXK = 256;
constexpr int CAT_LISTS_MAX = 32;    // candidate lists per user the re-rank kernel merges (splits x column sets)
constexpr int CAT_A_BLK = CAT_BM * CAT_BK * 2;                // 16 KB: one k-block of A
constexpr int CAT_B_TOTAL = 128 * 1024;                       // all B stages
constexpr int CAT_STAGE_WARPS = 8;                              // epilogue warps that own a 32x32 fp32 staging tile
constexpr int CAT_SMEM = CAT_KB_MAX * CAT_A_BLK + CAT_B_TOTAL + 1024 /*barriers*/ + CAT_STAGE_WARPS * 4096 + 1024 /*align*/;

struct CatGemmParams {
  int m_blocks;          // user blocks of CAT_BM * CG rows in this pass
  int m_pad;             // m_blocks * CAT_BM * CG
  int n_rows;            // valid user rows in this pass
  int n_split, tiles_per_split, n_tiles, k_blocks;
  const int32_t* keff;         // [m_pad] K_eff of each row: K + its listed recipes in this table, <= CAT_MAXK
  int boot_tiles;        // tiles of the bootstrap pass that seeds the thresholds (0: none); chunks recorded must fit a list
  int dense_min;         // rows of a warp with a hit in a chunk from which the per-lane (shared staging) resolution is used
  int a_split;           // 1: A = bf16 head + bf16 tail (two MMAs per B block; needs 2*k_blocks <= CAT_KB_MAX)
  int debug_mode;        // 0 = normal.  Ceiling measurements (results invalid; env FOODREC_CATALOG_DEBUG): 1 = epilogue only
                         // drains TMEM, 2 = accumulators never read (TMA+MMA alone), 3 = threshold +inf (filter fast path only)
  const int32_t* tile_group;   // [n_tiles] mask of each tile
  const int32_t* tile_valid;   // [n_tiles] recipes in the tile (256 except a group's last tile)
  const int32_t* block_first;  // [m_blocks] mask group a user block sweeps first (nullable: natural order)
  int group_lo[16], group_hi[16];   // tile range of each mask group
  int group_last_valid[16];         // recipes in the last tile of each group (the others are full)
  const float* bias;           // [16][m_pad]
  const float* margin2;        // [m_pad]  2E
  float* cand_sc;              // [n_split*NSET*m_pad][CAT_CAP] approx total score
  int32_t* cand_row;           // same shape: padded recipe row
  int32_t* cand_cnt;           // [n_split*NSET*m_pad]
  int32_t* ovf;                // [m_pad] 1 = candidate list overflowed
  unsigned long long* dbg;     // nullable: cycle counters {mma total, wait tempty, wait full, n, epi total, wait tfull, n}
#ifdef FR_CAT_TILE_BOUND
  // Per-tile error bound: E[u,t] = 0.5 * (margin2[u] * tile_rho[t] + margin2r[u]); the lists hold LOWER bounds
  // s_hat - E[u,t] and a recipe is kept iff its upper bound s_hat + E[u,t] reaches the K-th largest lower bound so far
  // (oracle/catalog_filter_model.py states and tests the rule).
  const float* tile_rho;       // [n_tiles] largest recipe norm of the tile / largest of the catalog, rounded up, <= 1
  const float* margin2r;       // [m_pad]  the part of 2E that does not scale with the recipe norm (fp32 roundings)
  int bn_shift;                // log2(tile width): padded recipe row -> tile
#endif
};

void launch_catalog_gemm(int cta_group, int epi_sets, int tile_n, int sm_count, const CUtensorMap& tmA, const CUtensorMap& tmB,
                         const CatGemmParams& p, cudaStream_t st);
cudaError_t catalog_gemm_configure();   // opt-in dynamic shared memory for both variants

// order-preserving float <-> uint32 key
__device__ __forceinline__ uint32_t fkey(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float funkey(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

}  // namespace fr
