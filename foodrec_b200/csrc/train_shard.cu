// Helper kernels of the row-sharded training step (one process per GPU):
//   P is sharded by user % W (samples are routed to the user owner when they are loaded),
//   R by recipe % W.  A rank requests the recipe rows its batch needs, the owners answer
//   (all-to-all over NVLink), and finished gradient rows travel the other way.
// Everything here is index bookkeeping; the row movers are the kernels of train_fwd.cu /
// train_seg.cu, pointed at the receive buffer (R := rbuf, items := slot ids).
#include "common.cuh"
#include "train.cuh"

namespace fr {

// owner-major key: sorting rows by it groups the unique recipes by owner, contiguously
__global__ void shard_prep_kernel(const ShardPlanParams p) {
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < p.S; r += gridDim.x * blockDim.x) {
    const uint32_t it = (uint32_t)p.items[r];
    p.okeys[r] = (it % (uint32_t)p.W) * p.items_per_rank + it / (uint32_t)p.W;
    p.cats_row[r] = p.cats_in ? p.cats_in[r] : __ldg(p.item_cats + it);
  }
}

__global__ void shard_heads_kernel(const ShardPlanParams p) {
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < p.S; q += gridDim.x * blockDim.x) {
    const uint32_t k = p.okeys_sorted[q];
    const bool head = q == 0 || p.okeys_sorted[q - 1] != k;
    p.flags[q] = head ? 1u : 0u;
    if (head) atomicAdd(p.owner_counts + k / p.items_per_rank, 1u);   // integer: order-independent
  }
}

// unique recipe k (rank of its run) of owner o gets slot o*cap + (k - start[o]); its request
// (the row index AT the owner) goes to req[slot]; every row learns its slot.
__global__ void shard_fill_kernel(const ShardPlanParams p) {
  uint32_t start[9];
  start[0] = 0;
  for (int o = 0; o < p.W && o < 8; ++o) start[o + 1] = start[o] + p.owner_counts[o];
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < p.S; q += gridDim.x * blockDim.x) {
    const uint32_t key = p.okeys_sorted[q];
    const uint32_t k = p.excl[q] + p.flags[q] - 1u;
    const uint32_t o = key / p.items_per_rank;
    const uint32_t j = k - start[o];
    uint32_t slot = o * (uint32_t)p.cap + j;
    if (j >= (uint32_t)p.cap) { p.out[FR_OUT_OVERFLOW] = 2.f; slot = o * (uint32_t)p.cap; }   // reported, never OOB
    else if (p.flags[q]) p.req[slot] = (int32_t)(key - o * p.items_per_rank);
    p.slot_of_row[p.perm[q]] = (int32_t)slot;
    p.slot_sorted[q] = slot;
  }
}

static int lin_grid(int64_t n, int sm_count) {
  int64_t g = (n + 255) / 256;
  if (g > (int64_t)sm_count * 8) g = (int64_t)sm_count * 8;
  return g < 1 ? 1 : (int)g;
}
void launch_shard_prep(const ShardPlanParams& p, const Launch& l) {
  shard_prep_kernel<<<lin_grid(p.S, l.sm_count), 256, 0, l.st>>>(p); ++g_launches;
}
void launch_shard_heads(const ShardPlanParams& p, const Launch& l) {
  shard_heads_kernel<<<lin_grid(p.S, l.sm_count), 256, 0, l.st>>>(p); ++g_launches;
}
void launch_shard_fill(const ShardPlanParams& p, const Launch& l) {
  shard_fill_kernel<<<lin_grid(p.S, l.sm_count), 256, 0, l.st>>>(p); ++g_launches;
}

// owner side: requests received from every rank -> sort keys (empty slots sort last)
__global__ void serve_keys_kernel(const int32_t* __restrict__ rreq, uint32_t n, uint32_t items_per_rank,
                                  uint32_t* __restrict__ keys, uint32_t* __restrict__ n_valid) {
  uint32_t cnt = 0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int32_t id = rreq[i];
    keys[i] = id < 0 ? items_per_rank : (uint32_t)id;
    cnt += id >= 0;
  }
  cnt = __reduce_add_sync(FR_FULL, cnt);
  if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(n_valid, cnt);
}
void launch_serve_keys(const int32_t* rreq, uint32_t n, uint32_t items_per_rank, uint32_t* keys, uint32_t* n_valid,
                       const Launch& l) {
  cudaMemsetAsync(n_valid, 0, sizeof(uint32_t), l.st);
  serve_keys_kernel<<<lin_grid(n, l.sm_count), 256, 0, l.st>>>(rreq, n, items_per_rank, keys, n_valid); ++g_launches;
}

// one warp per requested row; an empty request yields a zero row (staged path).  With peers the row of request slot
// (source s, j) is stored straight into rank s's receive buffer over NVLink (fused gather + exchange).
// bf16: 0 fp32 table, 1 bf16 table widened to fp32 rows, 2 bf16 table copied as stored (bf16 rows; staged path only).
__global__ void __launch_bounds__(FR_THREADS)
gather_rows_kernel(const float4* __restrict__ R, const int32_t* __restrict__ rreq, uint32_t n, int DV,
                   float4* __restrict__ out, const PeerPtrs peers, uint32_t n_table, int bf16) {
  const int lane = threadIdx.x & 31;
  const uint32_t gw = blockIdx.x * FR_WARPS_PER_BLOCK + (threadIdx.x >> 5), nw = gridDim.x * FR_WARPS_PER_BLOCK;
  for (uint32_t r = gw; r < n; r += nw) {
    const int32_t id = rreq[r];
    if (bf16 == 2) {
      uint2* d2 = tab_at<true>(out, (size_t)r * DV);
      for (int i = lane; i < DV; i += 32)
        d2[i] = (uint32_t)id >= n_table ? make_uint2(0u, 0u) : __ldg(tab_at<true>(R, (size_t)id * DV + i));
      continue;
    }
    float4* dst = out + (size_t)r * DV;
    if (peers.world > 0) {
      const uint32_t s = r / (uint32_t)peers.cap, j = r % (uint32_t)peers.cap;
      dst = peers.dst[s] + ((size_t)peers.rank * peers.cap + j) * DV;
    }
    if (id < 0 && peers.world > 0) continue;          // empty request slot: the consumer never reads it -- no store over NVLink
    for (int i = lane; i < DV; i += 32)
      dst[i] = (uint32_t)id >= n_table ? f4zero()                                  // (never out of the table)
               : (bf16 ? tab_ld_ro(tab_at<true>(R, (size_t)id * DV + i)) : R[(size_t)id * DV + i]);   // bf16 table -> fp32 row
  }
}
void launch_gather_rows(const float4* R, const int32_t* rreq, uint32_t n, int DV, float4* out, const PeerPtrs& peers,
                        const Launch& l, uint32_t n_table, int bf16) {
  if (n == 0) return;
  int grid = (int)((n + FR_WARPS_PER_BLOCK - 1) / FR_WARPS_PER_BLOCK);
  if (grid > l.sm_count * 16) grid = l.sm_count * 16;
  gather_rows_kernel<<<grid, FR_THREADS, 0, l.st>>>(R, rreq, n, DV, out, peers, n_table, bf16); ++g_launches;
}

// ---- routing of an UN-routed batch: a rank received arbitrary users; every group (sample / BPR triple) must reach
// the rank that owns its user (user % W).  Groups are bucketed by owner in batch order (stable sort by user % W),
// written front-packed into one fixed-capacity block per destination -- [rcap local user rows | rcap*group recipe
// ids | (pointwise) rcap labels], -1 padded -- exchanged with ONE all-to-all, and compacted in (source, position)
// order at the receiver.
__global__ void route_keys_kernel(const int32_t* __restrict__ users, int B, int W, uint32_t* __restrict__ keys,
                                  uint32_t* __restrict__ owner_counts) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B; i += gridDim.x * blockDim.x) {
    const uint32_t o = (uint32_t)users[i] % (uint32_t)W;
    keys[i] = o;
    atomicAdd(owner_counts + o, 1u);                      // integer: order-independent
  }
}
__global__ void route_fill_kernel(const int32_t* __restrict__ users, const int32_t* __restrict__ items,
                                  const float* __restrict__ labels, int B, int W, int group, int rcap,
                                  const uint32_t* __restrict__ okeys_sorted, const uint32_t* __restrict__ perm,
                                  const uint32_t* __restrict__ owner_counts, int32_t* __restrict__ send, float* __restrict__ flag) {
  uint32_t start[9]; start[0] = 0;
  for (int o = 0; o < W && o < 8; ++o) start[o + 1] = start[o] + owner_counts[o];
  const int blk = rcap * (1 + group + (labels ? 1 : 0));
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < B; q += gridDim.x * blockDim.x) {
    const uint32_t o = okeys_sorted[q], src = perm[q];
    const uint32_t j = (uint32_t)q - start[o];
    if (j >= (uint32_t)rcap) { *flag = 2.f; continue; }   // capacity of a (source, destination) pair exceeded
    int32_t* b = send + (size_t)o * blk;
    b[j] = users[src] / W;                                // LOCAL row at the owner
    for (int g = 0; g < group; ++g) b[rcap + j * group + g] = items[src * group + g];
    if (labels) b[rcap + rcap * group + j] = __float_as_int(labels[src]);
  }
}
// receiver: blocks are front-packed; count the valid groups of every source, then gather in (source, position) order
__global__ void route_count_kernel(const int32_t* __restrict__ recv, int W, int blk, int rcap, uint32_t* __restrict__ counts) {
  const int s = blockIdx.x;
  uint32_t c = 0;
  for (int j = threadIdx.x; j < rcap; j += blockDim.x) c += recv[(size_t)s * blk + j] >= 0;
  c = __reduce_add_sync(FR_FULL, c);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(counts + s, c);
}
__global__ void route_gather_kernel(const int32_t* __restrict__ recv, int W, int blk, int rcap, int group, int has_labels,
                                    const uint32_t* __restrict__ counts, int cap_out, int32_t* __restrict__ users,
                                    int32_t* __restrict__ items, float* __restrict__ labels, int32_t* __restrict__ n_out,
                                    float* __restrict__ flag) {
  uint32_t start[9]; start[0] = 0;
  for (int s = 0; s < W && s < 8; ++s) start[s + 1] = start[s] + counts[s];
  if (blockIdx.x == 0 && threadIdx.x == 0) { *n_out = (int32_t)min(start[W], (uint32_t)cap_out); if (start[W] > (uint32_t)cap_out) *flag = 2.f; }
  for (int s = 0; s < W; ++s) {
    const int32_t* b = recv + (size_t)s * blk;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < counts[s]; j += gridDim.x * blockDim.x) {
      const uint32_t d = start[s] + j;
      if (d >= (uint32_t)cap_out) continue;
      users[d] = b[j];
      for (int g = 0; g < group; ++g) items[d * group + g] = b[rcap + j * group + g];
      if (has_labels) labels[d] = __int_as_float(b[rcap + rcap * group + j]);
    }
  }
}
void launch_route_keys(const int32_t* users, int B, int W, uint32_t* keys, uint32_t* owner_counts, const Launch& l) {
  route_keys_kernel<<<lin_grid(B, l.sm_count), 256, 0, l.st>>>(users, B, W, keys, owner_counts); ++g_launches;
}
void launch_route_fill(const int32_t* users, const int32_t* items, const float* labels, int B, int W, int group, int rcap,
                       const uint32_t* okeys_sorted, const uint32_t* perm, const uint32_t* owner_counts, int32_t* send,
                       float* flag, const Launch& l) {
  route_fill_kernel<<<lin_grid(B, l.sm_count), 256, 0, l.st>>>(users, items, labels, B, W, group, rcap, okeys_sorted, perm,
                                                             owner_counts, send, flag); ++g_launches;
}
void launch_route_unpack(const int32_t* recv, int W, int blk, int rcap, int group, int has_labels, uint32_t* counts, int cap_out,
                         int32_t* users, int32_t* items, float* labels, int32_t* n_out, float* flag, const Launch& l) {
  cudaMemsetAsync(counts, 0, 8 * sizeof(uint32_t), l.st);
  route_count_kernel<<<W, 256, 0, l.st>>>(recv, W, blk, rcap, counts);
  route_gather_kernel<<<lin_grid(rcap, l.sm_count), 256, 0, l.st>>>(recv, W, blk, rcap, group, has_labels, counts, cap_out, users,
                                                                    items, labels, n_out, flag);
  g_launches += 2;
}

__global__ void add_inplace_kernel(float4* __restrict__ dst, const float4* __restrict__ src, int64_t n4) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x)
    dst[i] = add4(dst[i], src[i]);
}
void launch_add_inplace(float4* dst, const float4* src, int64_t n4, const Launch& l) {
  add_inplace_kernel<<<lin_grid(n4, l.sm_count), 256, 0, l.st>>>(dst, src, n4); ++g_launches;
}

}  // namespace fr
