// kernels_coal.cu -- log-prior of every tree's node times under the exponential-growth coalescent (sm_100a).
//
// Population size N(t) = n0 exp(g (t - t0)), times growing toward the present (a parent is never later than its children).  Read
// backwards in time, every tip (a sampling event) adds a lineage and every inner node (a coalescence) removes one, so with the events
// of a tree in ascending time order the number of lineages on (t_i, t_{i+1}) is k_i = 1 + #inner - #tips among events 0..i (1 above
// the root, where C(1, 2) = 0).  The log-density is
//   sum over coalescences c of -log N(t_c)  -  sum over intervals (a, b) of C(k, 2) * integral_a^b dt / N(t),
//   integral_a^b dt / N(t) = exp(-g (a - t0)) / n0 * (-expm1(-g (b - a)) / g)      (b - a when g (b - a) == 0),
// which is exact at g = 0 and loses nothing to cancellation for tiny |g|.  An interval of zero length contributes nothing, so tied
// times give the same value whatever order the sort leaves them in.
//
// Stages (all on the ctx stream):
//   1. one stable radix sort of every node position of the forest by time, 2. (forests of several trees) a stable radix sort of the
//   result by tree index: each tree's events then fill its own range of positions [node_base, node_base + num_nodes) in time order,
//   3. per forest tile of kTile sorted events: the sum of the lineage deltas, 4. an exclusive scan of those sums, 5. per tile: the
//   lineage count of every interval (block scan + the tile's carry) and its terms, summed, 6. per tree: the sum of its tiles' sums in
//   tile order (deterministic).
#include "dphy_internal.h"
#include "device_utils.cuh"

#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <cmath>

namespace dphy {

namespace {

struct CoalParams {
  double log_n0, inv_n0, g, t0;
};

__device__ __forceinline__ int tree_of_position(const ForestDev& f, int p) {
  int lo = 0, hi = f.num_trees - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (f.trees[mid].node_base <= p) lo = mid; else hi = mid - 1;
  }
  return lo;
}

__global__ void coal_iota_kernel(int32_t* __restrict__ pos, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) pos[i] = i;
}

__global__ void coal_tree_keys_kernel(ForestDev f, const int32_t* __restrict__ ev, int32_t* __restrict__ key) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < f.num_nodes) key[i] = tree_of_position(f, ev[i]);
}

// sorted event i of the tile this CTA covers: its index (or -1 past the tree's end) and the index one past the tree's last event
__device__ __forceinline__ int tile_event(const ForestDev& f, int tile, int* end) {
  const TreeDev T = f.trees[f.tile_tree[tile]];
  const int i = T.node_base + (tile - T.first_tile) * kTile + (int)threadIdx.x;
  *end = T.node_base + T.num_nodes;
  return i < *end ? i : -1;
}

__device__ __forceinline__ int lineage_delta(const ForestDev& f, int p) { return f.subtree_size[p] == 1 ? -1 : 1; }

__global__ void __launch_bounds__(kTile) coal_tile_delta_kernel(ForestDev f, const int32_t* __restrict__ ev, int32_t* __restrict__ tile_sum) {
  __shared__ int s_ws[kTile / 32];
  int end;
  const int i = tile_event(f, blockIdx.x, &end);
  const int s = block_sum<int, kTile>(i >= 0 ? lineage_delta(f, ev[i]) : 0, s_ws);
  if (threadIdx.x == 0) tile_sum[blockIdx.x] = s;
}

__global__ void __launch_bounds__(kTile) coal_tile_terms_kernel(ForestDev f, const int32_t* __restrict__ ev, const int32_t* __restrict__ tile_pre,
                                                               CoalParams c, double* __restrict__ tile_part) {
  __shared__ int s_iws[kTile / 32];
  __shared__ double s_dws[kTile / 32];
  int end;
  const int i = tile_event(f, blockIdx.x, &end);
  const int p = i >= 0 ? ev[i] : 0;
  const int s = i >= 0 ? lineage_delta(f, p) : 0;
  int tot;
  const int incl = block_scan_incl<int, kTile>(s, s_iws, &tot);
  double term = 0.0;
  if (i >= 0) {
    const int first_tile = f.trees[f.tile_tree[blockIdx.x]].first_tile;
    const double k = (double)(1 + tile_pre[blockIdx.x] - tile_pre[first_tile] + incl);   // lineages on (t_i, t_{i+1})
    const double a = f.t[p];
    if (s > 0) term -= c.log_n0 + c.g * (a - c.t0);                                        // -log N(t_c)
    if (i + 1 < end && k >= 2.0) {
      const double b = f.t[ev[i + 1]];
      if (b > a) {
        const double d = b - a, gd = c.g * d;
        const double w = gd == 0.0 ? d : -expm1(-gd) / c.g;
        term -= 0.5 * k * (k - 1.0) * exp(-c.g * (a - c.t0)) * c.inv_n0 * w;
      }
    }
  }
  const double sum = block_sum<double, kTile>(term, s_dws);
  if (threadIdx.x == 0) tile_part[blockIdx.x] = sum;
}

__global__ void __launch_bounds__(kTile) coal_tree_sum_kernel(ForestDev f, const double* __restrict__ tile_part, double* __restrict__ out) {
  __shared__ double s_ws[kTile / 32];
  const TreeDev T = f.trees[blockIdx.x];
  double v = 0.0;
  for (int j = threadIdx.x; j < T.num_tiles; j += kTile) v += tile_part[T.first_tile + j];
  v = block_sum<double, kTile>(v, s_ws);
  if (threadIdx.x == 0) out[blockIdx.x] = v;
}

}  // namespace
}  // namespace dphy

using namespace dphy;

extern "C" {

int dphy_forest_log_coalescent_prior(dphy_ctx* ctx, dphy_forest* fo, double n0, double g, double t0, double* out) {
  if (!ctx || !fo || !out) return DPHY_ERR_INVALID_ARGUMENT;
  if (!(n0 > 0.0) || !std::isfinite(n0) || !std::isfinite(g) || !std::isfinite(t0))
    return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "coalescent prior: n0 must be finite and > 0, g and t0 finite");
  const int T = fo->h.num_trees, N = fo->h.num_nodes, tiles = fo->h.num_tiles;
  if (T == 0) return DPHY_OK;
  cudaSetDevice(ctx->device);
  const int tree_bits = bits_for(T - 1);
  // scratch: sorted times (discarded), event positions and their ping-pong copy, tree keys and theirs, per-tile sums / parts, the
  // scan's tile totals, the per-tree results; then CUB's own temporary storage
  size_t cub_bytes = 0, cub2_bytes = 0;
  DPHY_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const double*)nullptr, (double*)nullptr, (const int32_t*)nullptr,
                                                 (int32_t*)nullptr, N, 0, 64, ctx->stream));
  if (T > 1)
    DPHY_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, cub2_bytes, (const int32_t*)nullptr, (int32_t*)nullptr, (const int32_t*)nullptr,
                                                   (int32_t*)nullptr, N, 0, tree_bits, ctx->stream));
  Slab slab;
  const int b_ts = slab.reserve(sizeof(double) * N), b_ev = slab.reserve(sizeof(int32_t) * N), b_ev2 = slab.reserve(sizeof(int32_t) * N);
  const int b_key = slab.reserve(sizeof(int32_t) * N), b_key2 = slab.reserve(sizeof(int32_t) * N);
  const int b_tsum = slab.reserve(sizeof(int32_t) * tiles), b_tpart = slab.reserve(sizeof(double) * tiles);
  const int b_tt = slab.reserve(sizeof(int32_t) * (tiles / 8192 + 2)), b_out = slab.reserve(sizeof(double) * T);
  const int b_cub = slab.reserve(std::max(cub_bytes, cub2_bytes));
  DevBlock blk(ctx->stream);
  if (!blk.alloc(slab.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(coalescent prior)");
  char* d = blk.p;
  double* ts = slab.at<double>(d, b_ts);
  int32_t* ev = slab.at<int32_t>(d, b_ev); int32_t* ev2 = slab.at<int32_t>(d, b_ev2);
  int32_t* key = slab.at<int32_t>(d, b_key); int32_t* key2 = slab.at<int32_t>(d, b_key2);
  int32_t* tsum = slab.at<int32_t>(d, b_tsum); double* tpart = slab.at<double>(d, b_tpart); int32_t* tt = slab.at<int32_t>(d, b_tt);
  double* d_out = slab.at<double>(d, b_out); void* cub_tmp = slab.at<char>(d, b_cub);
  const unsigned nb = (unsigned)((N + 255) / 256);
  coal_iota_kernel<<<nb, 256, 0, ctx->stream>>>(ev2, N);
  // every CUB sort below is counted as one launch
  cudaError_t ce = cub::DeviceRadixSort::SortPairs(cub_tmp, cub_bytes, (const double*)fo->h.t, ts, (const int32_t*)ev2, ev, N, 0, 64, ctx->stream);
  ctx->launches += 2;
  if (ce == cudaSuccess && T > 1) {
    coal_tree_keys_kernel<<<nb, 256, 0, ctx->stream>>>(fo->h, ev, key);
    ce = cub::DeviceRadixSort::SortPairs(cub_tmp, cub2_bytes, (const int32_t*)key, key2, (const int32_t*)ev, ev2, N, 0, tree_bits, ctx->stream);
    std::swap(ev, ev2);
    ctx->launches += 2;
  }
  if (ce == cudaSuccess) {
    coal_tile_delta_kernel<<<tiles, kTile, 0, ctx->stream>>>(fo->h, ev, tsum);
    ++ctx->launches;
    ce = cudaGetLastError();
  }
  int st = check_cuda(ctx, ce, "coalescent prior: sort");
  if (st == DPHY_OK) st = launch_scan_i32(ctx, tsum, tiles, tt);
  if (st == DPHY_OK) {
    CoalParams c{std::log(n0), 1.0 / n0, g, t0};
    coal_tile_terms_kernel<<<tiles, kTile, 0, ctx->stream>>>(fo->h, ev, tsum, c, tpart);
    coal_tree_sum_kernel<<<T, kTile, 0, ctx->stream>>>(fo->h, tpart, d_out);
    ctx->launches += 2;
    st = check_cuda(ctx, cudaGetLastError(), "coalescent prior kernels");
  }
  if (st == DPHY_OK) st = check_cuda(ctx, cudaMemcpyAsync(out, d_out, sizeof(double) * T, cudaMemcpyDeviceToHost, ctx->stream), "coalescent prior D2H");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "coalescent prior");
  return st;
}

}  // extern "C"
