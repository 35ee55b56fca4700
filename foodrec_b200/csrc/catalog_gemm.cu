// catalog_gemm_kernel<CG>: the dense contraction of full-catalog scoring on tcgen05, with the
// running top-K filter fused into the TMEM epilogue (see catalog.cuh for the maths).
//
// One CTA (CG = 1) or one CTA pair (CG = 2, tcgen05 cta_group::2, M = 256) owns a block of
// users for a whole sweep over its split of the recipe tiles:
//   warp 0   TMA producer: B tiles (recipes, bf16, 128B-swizzled) stream through an mbarrier
//            ring; the A block (one mask's user vectors, all of K) is loaded only when the
//            sweep enters a new mask group and then stays in shared memory (A-stationary: the
//            L2->SM traffic is the B stream alone, 1/(128*CG) bytes per flop)
//   warp 1   one thread issues tcgen05.mma (128*CG x 256 x 16 per instruction) into one of two
//            256-column fp32 accumulator stages in TMEM, commits free the smem stage / publish
//            the accumulator
//   warp 2   TMEM allocation
//   warps 4.. epilogue, NSET sets of 4 warps; set e owns accumulator columns [e*256/NSET, ...):
//            a thread owns one user row of its column set for the whole sweep (threshold and
//            candidate count live in its registers): tcgen05.ld 32 columns (next chunk's load in
//            flight) -> max-tree -> one compare; only a chunk that holds a value >= threshold
//            takes the per-value push path.  A row whose candidate list is nearly full is
//            compacted by its warp (exact K-th largest by bitwise binary search with warp REDUX,
//            keep >= kth - 2E).  Several warps per scheduler hide the TMEM / ALU latencies.
// No score matrix is ever written: HBM traffic is B once per concurrent wave plus O(K log) candidates.
#include <algorithm>

#include "catalog.cuh"
#include "common.cuh"
#include "internal.h"
#include "tc05.cuh"

namespace fr {

template <int CG, int BN>
struct CatCfg {
  static constexpr int B_ROWS = BN / CG;                // recipe rows this CTA loads per stage
  static constexpr int B_STAGE = B_ROWS * CAT_BK * 2;   // bytes
  static constexpr int NS = CAT_B_TOTAL / B_STAGE;      // smem ring depth: 4..16
  static constexpr int NACC = 512 / BN;                 // accumulator stages in TMEM: 2 (BN=256) / 4 (BN=128)
};

// Sweep order of one user block: the tiles of its first group [lo, hi) come first, then every other
// tile in natural order (lo == hi: natural order).  Users are sorted by their best mask group
// (largest category term), so a block starts where its rows' final top-K mostly lives: the
// running thresholds are tight from the start and later groups almost never push.
__device__ __forceinline__ int sweep_tile(const int i, const int lo, const int hi) {
  const int len = hi - lo;
  if (i < len) return lo + i;
  const int r = i - len;
  return r < lo ? r : r + len;
}
// A sweep is preceded by a BOOTSTRAP over its first `boot` tiles: the epilogue only records the maximum of every
// 32-column chunk (no pushes).  K_eff distinct chunk maxima are K_eff distinct recipes, so the K_eff-th largest of them
// is a valid lower bound of the final K_eff-th best score (catalog.cuh: exclusion lists): the real sweep (which starts over at its first tile) begins with a
// threshold near the top 1 % instead of -inf and skips the steep part of the ramp-up (~5x fewer pushes on a
// 200k-recipe catalog for ~8 % more MMA work).  Extended index e in [0, boot + n): tile index = e < boot ? e : e - boot.
struct SweepRange { int i0, i1, lo, hi, boot; };
__device__ __forceinline__ int sweep_index(const SweepRange& r, const int e) { return r.i0 + (e < r.boot ? e : e - r.boot); }
__device__ __forceinline__ int sweep_len(const SweepRange& r) { return r.boot + (r.i1 - r.i0); }
// mask group of a tile from the 15 group ranges in the kernel parameters (constant bank): the sweep
// stays inside one group for thousands of tiles, so the range is cached in registers and the
// per-tile cost is two compares -- no global load sits on the critical path of a tile.
struct GroupCursor { int g, lo, hi; };
__device__ __forceinline__ void group_seek(GroupCursor& c, const CatGemmParams& p, const int t) {
  if (t >= c.lo && t < c.hi) return;
  for (int g = 1; g < 16; ++g)
    if (t >= p.group_lo[g] && t < p.group_hi[g]) { c.g = g; c.lo = p.group_lo[g]; c.hi = p.group_hi[g]; return; }
}
__device__ __forceinline__ SweepRange sweep_range(const CatGemmParams& p, const int sp, const int mb) {
  SweepRange r;
  r.i0 = sp * p.tiles_per_split;
  r.i1 = min(r.i0 + p.tiles_per_split, p.n_tiles);
  r.lo = r.hi = 0;
  r.boot = min(p.boot_tiles, (r.i1 - r.i0) / 2);
  if (r.boot < 4) r.boot = 0;
  if (p.n_split == 1 && p.block_first) {
    const int g = __ldg(p.block_first + mb);
    r.lo = p.group_lo[g]; r.hi = p.group_hi[g];
  }
  return r;
}

// Warp-collective compaction of lane L's candidate row: exact K_eff-th largest of its entries by
// bitwise binary search (warp REDUX per bit), keep everything >= kth - 2E.  Returns lane L's new
// (count, threshold); every other lane gets its own values back.
struct CompactOut { int cnt; float thr; };
__device__ __noinline__ CompactOut catalog_warp_compact(const int L, const int lane, float* __restrict__ cand_sc,
                                                        int32_t* __restrict__ cand_row, const size_t my_base,
                                                        const int my_cnt, const float my_thr, const float my_margin2,
                                                        const int my_K, int32_t* ovf_flag, const bool drop_all
#ifdef FR_CAT_TILE_BOUND
                                                        , const float my_margin2r, const float* __restrict__ tile_rho,
                                                        const int bn_shift
#endif
                                                        ) {
  constexpr int NV = CAT_CAP / 32;
  const size_t base = __shfl_sync(FR_FULL, (unsigned long long)my_base, L);
  const int n = min(__shfl_sync(FR_FULL, my_cnt, L), CAT_CAP);
  const float m2 = __shfl_sync(FR_FULL, my_margin2, L);
  const int K = __shfl_sync(FR_FULL, my_K, L);        // the row's K_eff (K + its listed recipes in this table)
  float sc[NV]; int32_t rw[NV]; uint32_t key[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int e = i * 32 + lane;
    const bool ok = e < n;
    sc[i] = ok ? __ldcg(cand_sc + base + e) : 0.f;
    rw[i] = ok ? __ldcg(cand_row + base + e) : -1;
    key[i] = ok ? fkey(sc[i]) : 0u;
  }
  uint32_t res = 0;
  for (int bit = 31; bit >= 0; --bit) {
    const uint32_t trial = res | (1u << bit);
    int c = 0;
#pragma unroll
    for (int i = 0; i < NV; ++i) c += (key[i] >= trial);
    c = __reduce_add_sync(FR_FULL, c);
    if (c >= K) res = trial;
  }
#ifdef FR_CAT_TILE_BOUND
  const float m2r = __shfl_sync(FR_FULL, my_margin2r, L);
  const float nthr = funkey(res);      // the entries are LOWER bounds: their K-th largest bounds the K-th best true score from below
#else
  const float nthr = __fsub_rd(funkey(res), m2);
#endif
  if (drop_all) {                      // bootstrap: the entries were chunk maxima, only the bound is kept
    CompactOut r{my_cnt, my_thr};
    if (lane == L) { r.cnt = 0; if (n >= K) r.thr = nthr; }
    return r;
  }
  int out = 0;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
#ifdef FR_CAT_TILE_BOUND
    // keep iff the entry's UPPER bound (lower bound + 2E of its own tile, rounded up) reaches the threshold
    const bool keep = (i * 32 + lane < n) &&
                      (__fadd_ru(__fmaf_ru(m2, __ldg(tile_rho + (rw[i] >> bn_shift)), sc[i]), m2r) >= nthr);
#else
    const bool keep = (i * 32 + lane < n) && (sc[i] >= nthr);
#endif
    const uint32_t bal = __ballot_sync(FR_FULL, keep);
    if (keep) {
      const int pos = out + __popc(bal & ((1u << lane) - 1u));
      __stcg(cand_sc + base + pos, sc[i]);
      __stcg(cand_row + base + pos, rw[i]);
    }
    out += __popc(bal);
  }
  __syncwarp();
  CompactOut r{my_cnt, my_thr};
  if (lane == L) {
    r.cnt = out; r.thr = nthr;
    if (out > CAT_CAP - 64) { *ovf_flag = 1; r.thr = __int_as_float(0x7f800000); }   // too many near-ties: exact fallback
  }
  return r;
}

// Per-lane filter state of one (column set, user row): lives in registers for the whole sweep.
struct RowState {
  float thr, adj, bias, m2;
#ifdef FR_CAT_TILE_BOUND
  float m2r, er, bt;       // rounding part of 2E; E of (row, current tile); bias - E: what is added to a stored value
#define FR_CAT_SBIAS(s) ((s).bt)
#define FR_CAT_ADJ(s) __fsub_rd(__fsub_rd((s).thr, (s).bias), (s).er)            /* push iff v + bias + E >= thr */
#define FR_CAT_COMPACT_EXTRA(s, p) , (s).m2r, (p).tile_rho, (p).bn_shift
#else
#define FR_CAT_SBIAS(s) ((s).bias)
#define FR_CAT_ADJ(s) __fsub_rd((s).thr, (s).bias)
#define FR_CAT_COMPACT_EXTRA(s, p)
#endif
  int cnt, K;              // K = the row's K_eff (catalog.cuh: exclusion lists widen the filter)
  size_t base;
  int32_t* ovf;
};

// One 32-column chunk of the accumulator rows held by this warp (lane = user row).
// Fast path: 3-level max tree, one vote.  A chunk in which some row has a value >= its threshold is
// resolved with WARP-UNIFORM control flow only (per-element divergent branches cost a
// BSSY/BSYNC pair each and dominated the first version of this kernel): REDUX.OR finds the
// 8-column groups, then the columns, that hold a hit in any row; each such column is re-read
// from TMEM with a one-column tcgen05.ld (uniform address) and pushed under a predicate.
__device__ __forceinline__ void catalog_filter_chunk(const float (&v)[32], const uint32_t tchunk, const int col,
                                                     const int nvalid, const int n0, RowState& s,
                                                     const CatGemmParams& p, const int lane, float* stage, const bool boot) {
  float m[16], g8[4];
#pragma unroll
  for (int j = 0; j < 16; ++j) m[j] = fmaxf(v[2 * j], v[2 * j + 1]);
#pragma unroll
  for (int j = 0; j < 4; ++j) g8[j] = fmaxf(fmaxf(m[4 * j], m[4 * j + 1]), fmaxf(m[4 * j + 2], m[4 * j + 3]));
  const float mx = fmaxf(fmaxf(g8[0], g8[1]), fmaxf(g8[2], g8[3]));
  if (boot) {                                    // bootstrap pass: one value per chunk, no candidates
    if (col + 32 <= nvalid && s.thr < __int_as_float(0x7f800000)) {
      __stcg(p.cand_sc + s.base + s.cnt, mx + FR_CAT_SBIAS(s));
      ++s.cnt;
    }
    return;
  }
  if (!__any_sync(FR_FULL, mx >= s.adj)) return;
  // From here on the compiler may spill / the compaction call may save registers: the prefetched
  // chunk (an asynchronous tcgen05.ld into registers) must have landed before that can happen.
  tc::tmem_ld_wait();
#if !defined(FR_CAT_REREAD)
  // Dense regime (threshold ramp-up: several rows of the warp have hits in this chunk): every lane
  // resolves its own row.  The chunk is parked in a conflict-free [column][lane] shared tile so a lane
  // can index its values dynamically; the hit mask is built branch-free and popped bit by bit.
  if (stage != nullptr && __popc(__ballot_sync(FR_FULL, mx >= s.adj)) >= p.dense_min) {
    uint32_t hm = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      stage[j * 32 + lane] = v[j];
      hm |= (v[j] >= s.adj) ? (1u << j) : 0u;
    }
    if (col + 32 > nvalid) hm &= (nvalid > col) ? ((1u << (nvalid - col)) - 1u) : 0u;   // zero padding is never a candidate
    while (hm) {                                         // cnt <= CAP - 32 on entry (compaction policy): no bound check
      const int j = __ffs(hm) - 1;
      hm &= hm - 1;
      __stcg(p.cand_sc + s.base + s.cnt, stage[j * 32 + lane] + FR_CAT_SBIAS(s));
      __stcg(p.cand_row + s.base + s.cnt, n0 + col + j);
      ++s.cnt;
    }
    __syncwarp();
  } else
  // Sparse regime: votes only (no REDUX / find-first-set / TMEM re-read in the dependency chain): every
  // test is a warp-uniform predicate, the registers are indexed statically
  {
#pragma unroll
  for (int G = 0; G < 4; ++G) {
    if (__any_sync(FR_FULL, g8[G] >= s.adj)) {
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) {
        const float x = v[8 * G + jj];
        const bool hit = (x >= s.adj) && (col + 8 * G + jj < nvalid);   // zero padding is never a candidate
        if (__any_sync(FR_FULL, hit)) {
          if (hit) {                                       // cnt <= CAP - 32 on entry (compaction policy): no bound check
            __stcg(p.cand_sc + s.base + s.cnt, x + FR_CAT_SBIAS(s));
            __stcg(p.cand_row + s.base + s.cnt, n0 + col + 8 * G + jj);
            ++s.cnt;
          }
        }
      }
    }
  }
  }
#else
  const uint32_t gm = (g8[0] >= s.adj ? 1u : 0u) | (g8[1] >= s.adj ? 2u : 0u) | (g8[2] >= s.adj ? 4u : 0u) |
                      (g8[3] >= s.adj ? 8u : 0u);
  const uint32_t gmw = __reduce_or_sync(FR_FULL, gm);
#pragma unroll
  for (int G = 0; G < 4; ++G) {
    if (gmw & (1u << G)) {                                   // uniform
      uint32_t cm = 0;
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) cm |= (v[8 * G + jj] >= s.adj) ? (1u << jj) : 0u;
      uint32_t cmw = __reduce_or_sync(FR_FULL, cm);
      while (cmw) {                                          // uniform: columns with a hit in some row
        const int jj = __ffs(cmw) - 1;
        cmw &= cmw - 1;
        const int c = col + 8 * G + jj;
        if (c < nvalid) {                                    // zero padding at the end of a mask group is never a candidate
          const float x = tc::tmem_ld_32x1(tchunk + 8 * G + jj);
          if (x >= s.adj) {                                  // cnt <= CAP - 32 on entry (compaction policy): no bound check
            __stcg(p.cand_sc + s.base + s.cnt, x + FR_CAT_SBIAS(s));
            __stcg(p.cand_row + s.base + s.cnt, n0 + c);
            ++s.cnt;
          }
        }
      }
    }
  }
#endif
  uint32_t need = __ballot_sync(FR_FULL, s.cnt > CAT_CAP - 32);
  while (need) {
    const int L = __ffs(need) - 1;
    need &= need - 1;
    const CompactOut o = catalog_warp_compact(L, lane, p.cand_sc, p.cand_row, s.base, s.cnt, s.thr, s.m2, s.K, s.ovf, false
                                              FR_CAT_COMPACT_EXTRA(s, p));
    s.cnt = o.cnt; s.thr = o.thr;
    s.adj = FR_CAT_ADJ(s);
  }
}

template <int CG, int NSET, int BN>
__global__ void __launch_bounds__(128 + 128 * NSET, 1)
catalog_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const CatGemmParams p) {
  using C = CatCfg<CG, BN>;
  constexpr int NACC = C::NACC;
  constexpr int CW = BN / NSET;      // accumulator columns per epilogue warp set
  constexpr int NCH = CW / 32;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + CAT_KB_MAX * CAT_A_BLK;
  uint64_t* full = reinterpret_cast<uint64_t*>(sB + CAT_B_TOTAL);
  uint64_t* empty = full + C::NS;
  uint64_t* tfull = empty + C::NS;
  uint64_t* tempty = tfull + NACC;
  uint64_t* a_empty = tempty + NACC;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(a_empty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = (CG == 2) ? tc::cluster_ctarank() : 0u;
  const bool leader = rank == 0;

  if (warp == 0 && lane == 0) { tc::tma_prefetch_desc(&tmA); tc::tma_prefetch_desc(&tmB); }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < C::NS; ++i) { tc::mbar_init(&full[i], CG); tc::mbar_init(&empty[i], 1); }
    for (int i = 0; i < NACC; ++i) { tc::mbar_init(&tfull[i], 1); tc::mbar_init(&tempty[i], 4 * NSET * CG); }
    tc::mbar_init(a_empty, 1);
    tc::fence_barrier_init();
  }
  if (CG == 2) tc::cluster_sync_all();      // both CTAs resident and initialised before the pair allocates
  if (warp == 2) { tc::tmem_alloc<CG>(tmem_ptr, 512); tc::tmem_relinquish<CG>(); }
  tc::fence_before_sync();
  if (CG == 2) tc::cluster_sync_all(); else __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr;

  const int n_units = p.m_blocks * p.n_split;
  const int cluster_id = blockIdx.x / CG, n_clusters = gridDim.x / CG;
  const int kbn = p.k_blocks;
  const int kan = p.a_split ? 2 * kbn : kbn;     // A blocks resident in shared memory

  if (warp == 0 && lane == 0) {
    // ================= TMA producer =================
    uint32_t stage = 0, phase = 0, a_loads = 0;
    for (int unit = cluster_id; unit < n_units; unit += n_clusters) {
      const int sp = unit / p.m_blocks, mb = unit % p.m_blocks;
      const SweepRange sr = sweep_range(p, sp, mb);
      int prev_g = -1;
      GroupCursor gc{0, 0, 0};
      for (int e = 0; e < sweep_len(sr); ++e) {
        const int t = sweep_tile(sweep_index(sr, e), sr.lo, sr.hi);
        group_seek(gc, p, t);
        const int g = gc.g;
        const bool loadA = g != prev_g;
        prev_g = g;
        if (loadA) { tc::mbar_wait(a_empty, (a_loads & 1u) ^ 1u); ++a_loads; }   // MMAs of the previous A are done
        for (int kb = 0; kb < kbn; ++kb) {
          tc::mbar_wait(&empty[stage], phase ^ 1u);
          uint32_t bytes = C::B_STAGE;
          if (loadA && kb == 0) bytes += kan * CAT_A_BLK;
          if (CG == 1) tc::mbar_arrive_expect_tx(&full[stage], bytes);
          else if (leader) tc::mbar_arrive_expect_tx(&full[stage], 2 * bytes);
          else tc::mbar_arrive_cluster(&full[stage], 0);
          if (loadA && kb == 0) {
            const int arow = g * p.m_pad + mb * (CAT_BM * CG) + rank * CAT_BM;
            for (int k2 = 0; k2 < kan; ++k2)      // split operand: blocks [0,kbn) = bf16 head, [kbn,2kbn) = bf16 tail
              tc::tma_load_2d<CG>(sA + k2 * CAT_A_BLK, &tmA, &full[stage], k2 * CAT_BK, arow);
          }
          tc::tma_load_2d<CG>(sB + stage * C::B_STAGE, &tmB, &full[stage], kb * CAT_BK,
                              t * BN + (int)rank * C::B_ROWS);
          if (++stage == C::NS) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1 && lane == 0 && leader) {
    // ================= MMA issuer (one thread of the leader CTA) =================
    constexpr uint32_t idesc = tc::umma_idesc_bf16(CAT_BM * CG, BN);
    uint32_t stage = 0, phase = 0, tcount = 0;
    long long dbg_tempty = 0, dbg_full = 0;
    const long long dbg_t0 = clock64();
    for (int unit = cluster_id; unit < n_units; unit += n_clusters) {
      const int sp = unit / p.m_blocks, mb = unit % p.m_blocks;
      const SweepRange sr = sweep_range(p, sp, mb);
      GroupCursor gc{0, 0, 0};
      const int elen = sweep_len(sr);
      for (int e = 0; e < elen; ++e, ++tcount) {
        const uint32_t as = tcount % NACC, aph = (tcount / NACC) & 1u;
        const int t = sweep_tile(sweep_index(sr, e), sr.lo, sr.hi);
        group_seek(gc, p, t);
        const int tn = sweep_tile(sweep_index(sr, e + 1), sr.lo, sr.hi);
        const bool a_last = (e + 1 == elen) || tn < gc.lo || tn >= gc.hi;
        const long long c0 = p.dbg ? clock64() : 0;
        tc::mbar_wait(&tempty[as], aph ^ 1u);          // epilogue drained this accumulator stage
        tc::fence_after_sync();
        if (p.dbg) dbg_tempty += clock64() - c0;
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < kbn; ++kb) {
          const long long c1 = p.dbg ? clock64() : 0;
          tc::mbar_wait(&full[stage], phase);
          tc::fence_after_sync();
          if (p.dbg) dbg_full += clock64() - c1;
          const uint64_t ad = tc::umma_desc_sw128(sA + kb * CAT_A_BLK);
          const uint64_t bd = tc::umma_desc_sw128(sB + stage * C::B_STAGE);
#pragma unroll
          for (int k = 0; k < CAT_BK / 16; ++k)      // +32 B per k16 step inside the swizzle atom (addr field is >>4)
            tc::mma_bf16<CG>(d_tmem, ad + 2u * k, bd + 2u * k, idesc, (kb | k) ? 1u : 0u);
          if (p.a_split) {                           // + (A - bf16(A)) . B : the user operand is exact to 2^-16
            const uint64_t al = tc::umma_desc_sw128(sA + (kbn + kb) * CAT_A_BLK);
#pragma unroll
            for (int k = 0; k < CAT_BK / 16; ++k) tc::mma_bf16<CG>(d_tmem, al + 2u * k, bd + 2u * k, idesc, 1u);
          }
          tc::mma_commit<CG>(&empty[stage]);
          if (kb == kbn - 1) {
            tc::mma_commit<CG>(&tfull[as]);
            if (a_last) tc::mma_commit<CG>(a_empty);
          }
          if (++stage == C::NS) { stage = 0; phase ^= 1u; }
        }
      }
    }
    if (p.dbg) {
      atomicAdd(p.dbg + 0, (unsigned long long)(clock64() - dbg_t0));
      atomicAdd(p.dbg + 1, (unsigned long long)dbg_tempty);
      atomicAdd(p.dbg + 2, (unsigned long long)dbg_full);
      atomicAdd(p.dbg + 3, 1ULL);
    }
  } else if (warp >= 4) {
    // ================= epilogue: running top-K filter =================
    // warp set e = (warp-4)/4 owns accumulator columns [e*CW, (e+1)*CW); a warp can only read the
    // TMEM lane quarter warp%4, so thread (q, lane) is user row q*32+lane for the whole sweep and
    // keeps one candidate list per column set.
    const int q = warp & 3, e = (warp - 4) >> 2;
    float* stage = (warp - 4 < CAT_STAGE_WARPS)
                       ? reinterpret_cast<float*>(sB + CAT_B_TOTAL + 1024) + (warp - 4) * 1024 : nullptr;
    const int r_in_blk = q * 32 + lane;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + e * CW;
    const float INF = __int_as_float(0x7f800000);
    uint32_t tcount = 0;
    long long dbg_tfull = 0;
    const long long dbg_e0 = clock64();
    for (int unit = cluster_id; unit < n_units; unit += n_clusters) {
      const int sp = unit / p.m_blocks, mb = unit % p.m_blocks;
      const SweepRange sr = sweep_range(p, sp, mb);
      const int grow = mb * (CAT_BM * CG) + (int)rank * CAT_BM + r_in_blk;
      const bool valid = grow < p.n_rows;
      const size_t list = (static_cast<size_t>(sp) * NSET + e) * p.m_pad + grow;
      RowState s;
      s.base = list * CAT_CAP; s.m2 = __ldg(p.margin2 + grow); s.K = __ldg(p.keff + grow); s.thr = (valid && p.debug_mode != 3) ? -INF : INF; s.cnt = 0; s.bias = 0.f;
      s.adj = s.thr; s.ovf = p.ovf + grow;
#ifdef FR_CAT_TILE_BOUND
      s.m2r = __ldg(p.margin2r + grow); s.er = 0.f; s.bt = 0.f;
#endif
      int cur_g = -1;
      GroupCursor gc{0, 0, 0};
      for (int e2 = 0; e2 < sweep_len(sr); ++e2, ++tcount) {
        const uint32_t as = tcount % NACC, aph = (tcount / NACC) & 1u;
        const bool boot = e2 < sr.boot;
        if (e2 == sr.boot && sr.boot > 0) {             // bootstrap done: K_eff-th largest chunk maximum of every row -> threshold
          for (int L = 0; L < 32; ++L) {
            const CompactOut o = catalog_warp_compact(L, lane, p.cand_sc, p.cand_row, s.base, s.cnt, s.thr, s.m2, s.K, s.ovf, true
                                                      FR_CAT_COMPACT_EXTRA(s, p));
            s.cnt = o.cnt; s.thr = o.thr;
          }
        }
        const int t = sweep_tile(sweep_index(sr, e2), sr.lo, sr.hi);
        group_seek(gc, p, t);
        const int g = gc.g;
        const int nvalid = (t == gc.hi - 1) ? p.group_last_valid[g] : BN;     // rows of this tile that hold a recipe
        if (g != cur_g) { cur_g = g; s.bias = __ldg(p.bias + (size_t)g * p.m_pad + grow); }
#ifdef FR_CAT_TILE_BOUND
        s.er = __fmaf_ru(0.5f * s.m2, __ldg(p.tile_rho + t), 0.5f * s.m2r);    // E[row, tile], rounded up
        s.bt = __fsub_rd(s.bias, s.er);
#endif
        s.adj = FR_CAT_ADJ(s);                          // push iff  v + bias (+ E) >= thr
        const long long c2 = p.dbg ? clock64() : 0;
        tc::mbar_wait(&tfull[as], aph);
        tc::fence_after_sync();
        if (p.dbg) dbg_tfull += clock64() - c2;
        const int n0 = t * BN;
        const uint32_t tcol = t_lane + as * BN;
        auto release = [&]() {                          // accumulator stage fully read by this warp
          tc::fence_before_sync();
          __syncwarp();
          if (lane == 0) { if (CG == 1) tc::mbar_arrive(&tempty[as]); else tc::mbar_arrive_cluster(&tempty[as], 0); }
        };
#if defined(FR_CAT_REREAD)
        auto release_early = [&]() {};
#else
        auto release_early = release;                   // the accumulator is in registers once its last load has landed
#endif
        if (p.debug_mode == 2) { release(); continue; }     // MMA/TMA ceiling: accumulators are never read
        if constexpr (NSET <= 2) {
          float va[32], vb[32];
          __syncwarp();
          tc::tmem_ld_32x32(tcol, va);
#pragma unroll 1
          for (int c = 0; c < NCH; c += 2) {            // TMEM load of chunk c+1 is in flight while chunk c is filtered
            tc::tmem_ld_wait();
            __syncwarp();
            if (c + 1 < NCH) tc::tmem_ld_32x32(tcol + (c + 1) * 32, vb); else release_early();
            if (p.debug_mode == 0 || p.debug_mode == 3) catalog_filter_chunk(va, tcol + c * 32, e * CW + c * 32, nvalid, n0, s, p, lane, stage, boot);
            else if (va[0] + va[13] + va[31] == 12345.f) s.cnt++;
            if (c + 1 < NCH) {
              tc::tmem_ld_wait();
              __syncwarp();
              if (c + 2 < NCH) tc::tmem_ld_32x32(tcol + (c + 2) * 32, va); else release_early();
              if (p.debug_mode == 0 || p.debug_mode == 3) catalog_filter_chunk(vb, tcol + (c + 1) * 32, e * CW + (c + 1) * 32, nvalid, n0, s, p, lane, stage, boot);
              else if (vb[0] + vb[13] + vb[31] == 12345.f) s.cnt++;
            }
          }
        } else {                                        // 16 epilogue warps: 96 registers each, no prefetch buffer
#pragma unroll
          for (int c = 0; c < NCH; ++c) {
            float va[32];
            __syncwarp();
            tc::tmem_ld_32x32(tcol + c * 32, va);
            tc::tmem_ld_wait();
            if (c == NCH - 1) release_early();
            if (p.debug_mode == 0 || p.debug_mode == 3) catalog_filter_chunk(va, tcol + c * 32, e * CW + c * 32, nvalid, n0, s, p, lane, stage, boot);
            else if (va[0] + va[13] + va[31] == 12345.f) s.cnt++;
          }
        }
#if defined(FR_CAT_REREAD)
        release();                                      // after the last possible re-read of this stage
#endif
      }
      if (valid) p.cand_cnt[list] = min(s.cnt, CAT_CAP);
    }
    if (p.dbg && lane == 0) {
      atomicAdd(p.dbg + 4, (unsigned long long)(clock64() - dbg_e0));
      atomicAdd(p.dbg + 5, (unsigned long long)dbg_tfull);
      atomicAdd(p.dbg + 6, 1ULL);
    }
  }

  __syncwarp();
  tc::fence_before_sync();
  if (CG == 2) tc::cluster_sync_all(); else __syncthreads();
  if (warp == 2) tc::tmem_dealloc<CG>(tmem_base, 512);
}

template <int CG, int NSET, int BN>
static cudaError_t configure_one() {
  return cudaFuncSetAttribute(catalog_gemm_kernel<CG, NSET, BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, CAT_SMEM);
}
template <int BN>
static cudaError_t configure_bn() {
  cudaError_t e;
  if ((e = configure_one<1, 1, BN>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 1, BN>()) != cudaSuccess) return e;
  if ((e = configure_one<1, 2, BN>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 2, BN>()) != cudaSuccess) return e;
  if ((e = configure_one<1, 4, BN>()) != cudaSuccess) return e;
  return configure_one<2, 4, BN>();
}
cudaError_t catalog_gemm_configure() {
  cudaError_t e = configure_bn<256>();
  if (e != cudaSuccess) return e;
  return configure_bn<128>();
}

template <int CG, int NSET, int BN>
static void launch_one(int sm_count, const CUtensorMap& tmA, const CUtensorMap& tmB, const CatGemmParams& p, cudaStream_t st) {
  const int n_units = p.m_blocks * p.n_split;
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(128 + 128 * NSET);
  cfg.dynamicSmemBytes = CAT_SMEM;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  const int clusters = std::max(1, std::min(sm_count / CG, n_units));
  cfg.gridDim = dim3(CG * clusters);
  if (CG == 2) {
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
  }
  cudaLaunchKernelEx(&cfg, catalog_gemm_kernel<CG, NSET, BN>, tmA, tmB, p);
  ++g_launches;
}

template <int BN>
static void launch_bn(int cta_group, int epi_sets, int sm_count, const CUtensorMap& tmA, const CUtensorMap& tmB,
                      const CatGemmParams& p, cudaStream_t st) {
  if (cta_group == 2) {
    if (epi_sets == 4) launch_one<2, 4, BN>(sm_count, tmA, tmB, p, st);
    else if (epi_sets == 2) launch_one<2, 2, BN>(sm_count, tmA, tmB, p, st);
    else launch_one<2, 1, BN>(sm_count, tmA, tmB, p, st);
  } else {
    if (epi_sets == 4) launch_one<1, 4, BN>(sm_count, tmA, tmB, p, st);
    else if (epi_sets == 2) launch_one<1, 2, BN>(sm_count, tmA, tmB, p, st);
    else launch_one<1, 1, BN>(sm_count, tmA, tmB, p, st);
  }
}

void launch_catalog_gemm(int cta_group, int epi_sets, int tile_n, int sm_count, const CUtensorMap& tmA,
                         const CUtensorMap& tmB, const CatGemmParams& p, cudaStream_t st) {
  if (tile_n == 128) launch_bn<128>(cta_group, epi_sets, sm_count, tmA, tmB, p, st);
  else launch_bn<256>(cta_group, epi_sets, sm_count, tmA, tmB, p, st);
}

}  // namespace fr
