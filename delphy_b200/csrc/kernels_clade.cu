// kernels_clade.cu -- clade support over forests of posterior trees and the maximum clade credibility score (sm_100a).
//
// Device order is a per-tree DFS pre-order, so the tips below the node at position p are the tips among positions [p, p + size(p)).
// Put every tip's two lane keys k_j(i) = splitmix64(i << 1 | j) (i: its host node index) at its position and 0 at inner nodes, and let
// S be their forest-wide exclusive prefix sum, wrapping per u64 lane.  The clade key of p is then S[p + size(p)] - S[p]: the prefix
// of the trees before p's cancels, so the scan needs no per-tree segments.
//
// dphy_clade_table_add:
//   1. the lane keys, the tip-set check (every tip's host index is in the table's bitmap; tips counted), the scan, the clade keys;
//   2. a stable radix sort of (key, t) by key over the whole forest, a run-length encoding of the sorted keys, and per run its length
//      and the sum of its times in sorted order -- the stable sort leaves them in tree order;
//   3. the number of the batch's clades the table already holds (binary search), so that the new table is allocated at its exact
//      size; a merge of table and batch, then equal neighbours added (each clade is at most once in either);
//   4. the new arrays swapped in.  Nothing of the table changes before step 4: a refusal or a failed allocation leaves it as it was.
// dphy_clade_table_score / _node_support: step 1, then a binary search of every node's key in the table.  The score sums log(count / T)
// per kTile-node tile and then the tree's tiles in order: a fixed association, so equal tables give bit-identical scores.
#include "dphy_internal.h"
#include "device_utils.cuh"

#include <cub/device/device_merge.cuh>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_reduce.cuh>
#include <cub/device/device_run_length_encode.cuh>
#include <cub/device/device_scan.cuh>
#include <cuda/std/tuple>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

namespace dphy {

// found by argument-dependent lookup inside CUB (run-length encoding, reduce by key)
__host__ __device__ __forceinline__ bool operator==(const CladeKey& a, const CladeKey& b) { return a.k0 == b.k0 && a.k1 == b.k1; }

namespace {

enum { kStBad = 0, kStTips = 1, kStRefTips = 2, kStKnown = 3, kStLen = 4 };   // status words of a call (device, zeroed per call)

__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  uint64_t z = x + 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}

struct CladeKeyLess {
  __host__ __device__ __forceinline__ bool operator()(const CladeKey& a, const CladeKey& b) const {
    return a.k0 < b.k0 || (a.k0 == b.k0 && a.k1 < b.k1);
  }
};
struct CladeKeyDecomposer {   // radix order == CladeKeyLess: k0 most significant
  __host__ __device__ ::cuda::std::tuple<uint64_t&, uint64_t&> operator()(CladeKey& k) const { return {k.k0, k.k1}; }
};
struct CladeKeyAdd {
  __host__ __device__ __forceinline__ CladeKey operator()(const CladeKey& a, const CladeKey& b) const { return {a.k0 + b.k0, a.k1 + b.k1}; }
};
struct CladeValAdd {          // at most two operands per clade (table, batch): IEEE addition of two is order-free
  __host__ __device__ __forceinline__ CladeVal operator()(const CladeVal& a, const CladeVal& b) const {
    return {a.count + b.count, a.t_sum + b.t_sum};
  }
};

struct TableView {
  const CladeKey* keys;
  const CladeVal* vals;
  int64_t n;
  double num_trees;
};

__device__ __forceinline__ int64_t find_clade(const CladeKey* __restrict__ keys, int64_t n, CladeKey k) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (CladeKeyLess{}(keys[mid], k)) lo = mid + 1; else hi = mid;
  }
  return lo < n && keys[lo] == k ? lo : -1;
}

__device__ __forceinline__ void count_warp(bool pred, unsigned long long* counter) {
  const unsigned m = __ballot_sync(0xffffffffu, pred);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(counter, (unsigned long long)__popc(m));
}

// first add: the tips of tree 0 (positions [0, n0)) define the table's tip set
__global__ void clade_tip_bitmap_kernel(ForestDev f, int n0, uint32_t* __restrict__ tips, unsigned long long* __restrict__ status) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const bool tip = p < n0 && f.subtree_size[p] == 1;
  if (tip) {
    const int id = f.node_id[p];
    atomicOr(&tips[id >> 5], 1u << (id & 31));
  }
  count_warp(tip, &status[kStRefTips]);
}

__global__ void clade_tip_keys_kernel(ForestDev f, const uint32_t* __restrict__ tips, CladeKey* __restrict__ key,
                                      unsigned long long* __restrict__ status) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const bool tip = p < f.num_nodes && f.subtree_size[p] == 1;
  bool bad = false;
  if (p < f.num_nodes) {
    CladeKey k{0, 0};
    if (tip) {
      const uint32_t id = (uint32_t)f.node_id[p];   // < N: every tree has the table's N nodes
      k.k0 = splitmix64((uint64_t)id << 1);
      k.k1 = splitmix64((uint64_t)id << 1 | 1u);
      bad = ((tips[id >> 5] >> (id & 31)) & 1u) == 0;
    }
    key[p] = k;
  }
  count_warp(tip, &status[kStTips]);
  count_warp(bad, &status[kStBad]);
}

// S[N + 1]: exclusive prefix of the lane keys
__global__ void clade_keys_kernel(ForestDev f, const CladeKey* __restrict__ S, CladeKey* __restrict__ h) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= f.num_nodes) return;
  const CladeKey a = S[p], b = S[p + f.subtree_size[p]];
  h[p] = CladeKey{b.k0 - a.k0, b.k1 - a.k1};
}

// per run of equal sorted keys: how many trees have the clade and the sum of its times, in tree order
__global__ void clade_run_sums_kernel(const int32_t* __restrict__ run_len, const int32_t* __restrict__ run_off, const double* __restrict__ ts,
                                      int num_runs, CladeVal* __restrict__ val) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= num_runs) return;
  const int o = run_off[r], c = run_len[r];
  double s = ts[o];
  for (int k = 1; k < c; ++k) s += ts[o + k];
  val[r] = CladeVal{c, s};
}

__global__ void clade_count_known_kernel(TableView tab, const CladeKey* __restrict__ bkey, int nb, unsigned long long* __restrict__ status) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  count_warp(r < nb && find_clade(tab.keys, tab.n, bkey[r]) >= 0, &status[kStKnown]);
}

__global__ void __launch_bounds__(kTile) clade_score_tile_kernel(ForestDev f, const CladeKey* __restrict__ h, TableView tab,
                                                                 double* __restrict__ tile_part) {
  __shared__ double s_ws[kTile / 32];
  const TreeDev T = f.trees[f.tile_tree[blockIdx.x]];
  const int i = T.node_base + (int)(blockIdx.x - T.first_tile) * kTile + (int)threadIdx.x;
  double term = 0.0;
  if (i < T.node_base + T.num_nodes) {
    const int64_t j = find_clade(tab.keys, tab.n, h[i]);
    term = j < 0 ? -INFINITY : log((double)tab.vals[j].count / tab.num_trees);
  }
  const double s = block_sum<double, kTile>(term, s_ws);
  if (threadIdx.x == 0) tile_part[blockIdx.x] = s;
}

__global__ void __launch_bounds__(kTile) clade_tree_sum_kernel(ForestDev f, const double* __restrict__ tile_part, double* __restrict__ out) {
  __shared__ double s_ws[kTile / 32];
  const TreeDev T = f.trees[blockIdx.x];
  double v = 0.0;
  for (int j = threadIdx.x; j < T.num_tiles; j += kTile) v += tile_part[T.first_tile + j];
  v = block_sum<double, kTile>(v, s_ws);
  if (threadIdx.x == 0) out[blockIdx.x] = v;
}

__global__ void clade_node_support_kernel(ForestDev f, int tree, const CladeKey* __restrict__ h, TableView tab, int64_t* __restrict__ count,
                                          double* __restrict__ mean_t) {
  const TreeDev T = f.trees[tree];
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= T.num_nodes) return;
  const int64_t j = find_clade(tab.keys, tab.n, h[T.node_base + f.pos_of_node[T.node_base + v]]);   // pos_of_node is tree-local
  if (j < 0) {
    count[v] = 0;
    mean_t[v] = NAN;
  } else {
    const CladeVal c = tab.vals[j];
    count[v] = c.count;
    mean_t[v] = c.t_sum / (double)c.count;
  }
}

unsigned blocks(int64_t n) { return (unsigned)((n + 255) / 256); }

// Every tree of `fo` must have N nodes (N = the table's, or tree 0's for a table that is still empty).
int check_sizes(dphy_ctx* ctx, const dphy_clade_table* tab, const dphy_forest* fo, int* N) {
  *N = tab->num_nodes >= 0 ? tab->num_nodes : fo->trees[0].num_nodes;
  for (const TreeDev& tr : fo->trees)
    if (tr.num_nodes != *N)
      return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "clade table: every tree must have " + std::to_string(*N) + " nodes, like the trees added before");
  return DPHY_OK;
}

bool tips_ok(const unsigned long long* st, int64_t num_trees, int64_t tips_per_tree) {
  return st[kStBad] == 0 && st[kStTips] == (unsigned long long)(num_trees * tips_per_tree);
}

// Scratch of one call: the status words, the scan, the clade key of every position of the forest, and `extra` bytes for the caller.
struct KeyScratch {
  explicit KeyScratch(cudaStream_t s) : blk(s) {}
  DevBlock blk;
  unsigned long long* status = nullptr;
  CladeKey* S = nullptr;   // [N + 1]; free for the caller once the keys are made
  CladeKey* h = nullptr;   // [N]
  char* extra = nullptr;
};

// Allocates ks and enqueues step 1 (lane keys + tip check, scan, clade keys).  tips == nullptr: the bitmap is built first, into the
// extra block's first `bitmap_words` words, from the tips of tree 0.
int clade_keys(dphy_ctx* ctx, dphy_forest* fo, const uint32_t* tips, int bitmap_words, size_t extra, KeyScratch& ks) {
  const int N = fo->h.num_nodes;
  size_t scan_bytes = 0;
  DPHY_CUDA(ctx, cub::DeviceScan::InclusiveScan(nullptr, scan_bytes, (const CladeKey*)nullptr, (CladeKey*)nullptr, CladeKeyAdd{}, N, ctx->stream));
  Slab slab;
  const int b_st = slab.reserve(sizeof(unsigned long long) * kStLen), b_S = slab.reserve(sizeof(CladeKey) * ((size_t)N + 1));
  const int b_h = slab.reserve(sizeof(CladeKey) * (size_t)N), b_cub = slab.reserve(scan_bytes), b_extra = slab.reserve(extra);
  if (!ks.blk.alloc(slab.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(clade table scratch)");
  char* d = ks.blk.p;
  ks.status = slab.at<unsigned long long>(d, b_st);
  ks.S = slab.at<CladeKey>(d, b_S);
  ks.h = slab.at<CladeKey>(d, b_h);
  ks.extra = slab.at<char>(d, b_extra);
  DPHY_CUDA(ctx, cudaMemsetAsync(ks.status, 0, sizeof(unsigned long long) * kStLen, ctx->stream));
  DPHY_CUDA(ctx, cudaMemsetAsync(ks.S, 0, sizeof(CladeKey), ctx->stream));
  if (!tips) {
    uint32_t* bm = (uint32_t*)ks.extra;
    DPHY_CUDA(ctx, cudaMemsetAsync(bm, 0, sizeof(uint32_t) * bitmap_words, ctx->stream));
    const int n0 = fo->trees[0].num_nodes;
    clade_tip_bitmap_kernel<<<blocks(n0), 256, 0, ctx->stream>>>(fo->h, n0, bm, ks.status);
    ++ctx->launches;
    tips = bm;
  }
  clade_tip_keys_kernel<<<blocks(N), 256, 0, ctx->stream>>>(fo->h, tips, ks.h, ks.status);
  DPHY_CUDA(ctx, cub::DeviceScan::InclusiveScan(slab.at<char>(d, b_cub), scan_bytes, (const CladeKey*)ks.h, ks.S + 1, CladeKeyAdd{}, N, ctx->stream));
  clade_keys_kernel<<<blocks(N), 256, 0, ctx->stream>>>(fo->h, ks.S, ks.h);
  ctx->launches += 3;
  return check_cuda(ctx, cudaGetLastError(), "clade keys");
}

int check_use(dphy_ctx* ctx, const dphy_clade_table* tab, const dphy_forest* fo) {
  if (!ctx || !tab || !fo) return DPHY_ERR_INVALID_ARGUMENT;
  if (tab->ctx != ctx) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "clade table: used with a ctx other than the one that made it");
  return DPHY_OK;
}

TableView view_of(const dphy_clade_table* tab) { return TableView{tab->d_keys, tab->d_vals, tab->num_clades, (double)tab->num_trees}; }

}  // namespace
}  // namespace dphy

using namespace dphy;

extern "C" {

int dphy_clade_table_create(dphy_ctx* ctx, dphy_clade_table** out) {
  if (!ctx || !out) return DPHY_ERR_INVALID_ARGUMENT;
  dphy_clade_table* t = new dphy_clade_table();
  t->ctx = ctx;
  *out = t;
  return DPHY_OK;
}

void dphy_clade_table_destroy(dphy_ctx* ctx, dphy_clade_table* tab) {
  if (!ctx || !tab) return;
  cudaSetDevice(ctx->device);
  if (tab->d_keys) cudaFreeAsync(tab->d_keys, ctx->stream);
  if (tab->d_tips) cudaFreeAsync(tab->d_tips, ctx->stream);
  cudaStreamSynchronize(ctx->stream);
  delete tab;
}

int dphy_clade_table_info(const dphy_clade_table* tab, int64_t* num_trees, int64_t* num_clades, int64_t* device_bytes) {
  if (!tab) return DPHY_ERR_INVALID_ARGUMENT;
  if (num_trees) *num_trees = tab->num_trees;
  if (num_clades) *num_clades = tab->num_clades;
  if (device_bytes) *device_bytes = (int64_t)tab->bytes;
  return DPHY_OK;
}

int dphy_clade_table_add(dphy_ctx* ctx, dphy_clade_table* tab, dphy_forest* fo) {
  int st = check_use(ctx, tab, fo);
  if (st != DPHY_OK) return st;
  const int T = fo->h.num_trees, N = fo->h.num_nodes;
  if (T == 0) return DPHY_OK;
  int Nt;
  if ((st = check_sizes(ctx, tab, fo, &Nt)) != DPHY_OK) return st;
  cudaSetDevice(ctx->device);
  const bool first = tab->num_nodes < 0;
  const int words = (Nt + 31) / 32;
  cudaStream_t s = ctx->stream;

  // ---- step 1 + 2: keys, sort, run-length encoding.  Extra scratch: [bitmap (first add)] sorted keys, sorted times, run lengths,
  // run offsets, the run count, CUB's storage.  The batch's unique keys go to S, its values to h (both dead by then).
  size_t sort_bytes = 0, rle_bytes = 0, off_bytes = 0;
  DPHY_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const CladeKey*)nullptr, (CladeKey*)nullptr, (const double*)nullptr,
                                                 (double*)nullptr, N, CladeKeyDecomposer{}, s));
  DPHY_CUDA(ctx, cub::DeviceRunLengthEncode::Encode(nullptr, rle_bytes, (const CladeKey*)nullptr, (CladeKey*)nullptr, (int32_t*)nullptr,
                                                    (int32_t*)nullptr, N, s));
  DPHY_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, off_bytes, (const int32_t*)nullptr, (int32_t*)nullptr, N, s));
  Slab ex;
  if (first) ex.reserve(sizeof(uint32_t) * words);    // the tip bitmap, at the block's start (clade_keys)
  const int b_hs = ex.reserve(sizeof(CladeKey) * (size_t)N), b_ts = ex.reserve(sizeof(double) * (size_t)N);
  const int b_len = ex.reserve(sizeof(int32_t) * (size_t)N), b_off = ex.reserve(sizeof(int32_t) * (size_t)N);
  const int b_nr = ex.reserve(sizeof(int32_t)), b_cub = ex.reserve(std::max(sort_bytes, std::max(rle_bytes, off_bytes)));
  KeyScratch ks(s);
  if ((st = clade_keys(ctx, fo, first ? nullptr : tab->d_tips, words, ex.total, ks)) != DPHY_OK) return st;
  CladeKey* hs = ex.at<CladeKey>(ks.extra, b_hs);
  double* ts = ex.at<double>(ks.extra, b_ts);
  int32_t* run_len = ex.at<int32_t>(ks.extra, b_len);
  int32_t* run_off = ex.at<int32_t>(ks.extra, b_off);
  int32_t* d_nruns = ex.at<int32_t>(ks.extra, b_nr);
  void* cub_tmp = ex.at<char>(ks.extra, b_cub);
  CladeKey* bkey = ks.S;
  CladeVal* bval = (CladeVal*)ks.h;
  DPHY_CUDA(ctx, cub::DeviceRadixSort::SortPairs(cub_tmp, sort_bytes, (const CladeKey*)ks.h, hs, (const double*)fo->h.t, ts, N,
                                                 CladeKeyDecomposer{}, s));
  DPHY_CUDA(ctx, cub::DeviceRunLengthEncode::Encode(cub_tmp, rle_bytes, (const CladeKey*)hs, bkey, run_len, d_nruns, N, s));
  ctx->launches += 5;
  unsigned long long hst[kStLen];
  int32_t nb = 0;
  DPHY_CUDA(ctx, cudaMemcpyAsync(hst, ks.status, sizeof(hst), cudaMemcpyDeviceToHost, s));
  DPHY_CUDA(ctx, cudaMemcpyAsync(&nb, d_nruns, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  DPHY_CUDA(ctx, cudaStreamSynchronize(s));
  const int64_t tips_per_tree = first ? (int64_t)hst[kStRefTips] : tab->num_tips;
  if (!tips_ok(hst, T, tips_per_tree))
    return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "clade table: every tree must have the same tips (host node indices) as the trees added before");

  // per run: count and time sum (tree order); how many of the batch's clades the table holds already
  DPHY_CUDA(ctx, cub::DeviceScan::ExclusiveSum(cub_tmp, off_bytes, (const int32_t*)run_len, run_off, nb, s));
  clade_run_sums_kernel<<<blocks(nb), 256, 0, s>>>(run_len, run_off, ts, nb, bval);
  ctx->launches += 2;
  const int64_t nt = tab->num_clades;
  if (nt > 0) {
    clade_count_known_kernel<<<blocks(nb), 256, 0, s>>>(view_of(tab), bkey, nb, ks.status);
    ++ctx->launches;
    DPHY_CUDA(ctx, cudaMemcpyAsync(&hst[kStKnown], &ks.status[kStKnown], sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
  }
  DPHY_CUDA(ctx, cudaGetLastError());
  DPHY_CUDA(ctx, cudaStreamSynchronize(s));
  const int64_t n_new = nt + nb - (int64_t)hst[kStKnown];
  if (nt + nb > (int64_t)INT32_MAX)
    return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "clade table: more than 2^31 - 1 clades");

  // ---- step 3: the new table at its exact size
  Slab tbl;
  const int t_keys = tbl.reserve(sizeof(CladeKey) * (size_t)n_new), t_vals = tbl.reserve(sizeof(CladeVal) * (size_t)n_new);
  DevBlock table_blk(s);
  if (!table_blk.alloc(tbl.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(clade table)");
  CladeKey* new_keys = tbl.at<CladeKey>(table_blk.p, t_keys);
  CladeVal* new_vals = tbl.at<CladeVal>(table_blk.p, t_vals);
  DevBlock tips_blk(s);
  if (first) {
    if (!tips_blk.alloc(sizeof(uint32_t) * words)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(clade table tips)");
    DPHY_CUDA(ctx, cudaMemcpyAsync(tips_blk.p, ks.extra, sizeof(uint32_t) * words, cudaMemcpyDeviceToDevice, s));
  }
  int32_t n_out = nb;
  if (nt == 0) {
    DPHY_CUDA(ctx, cudaMemcpyAsync(new_keys, bkey, sizeof(CladeKey) * nb, cudaMemcpyDeviceToDevice, s));
    DPHY_CUDA(ctx, cudaMemcpyAsync(new_vals, bval, sizeof(CladeVal) * nb, cudaMemcpyDeviceToDevice, s));
  } else {
    const int m = (int)(nt + nb);
    size_t merge_bytes = 0, rbk_bytes = 0;
    DPHY_CUDA(ctx, cub::DeviceMerge::MergePairs(nullptr, merge_bytes, (const CladeKey*)nullptr, (const CladeVal*)nullptr, (int)nt,
                                                (const CladeKey*)nullptr, (const CladeVal*)nullptr, nb, (CladeKey*)nullptr, (CladeVal*)nullptr,
                                                CladeKeyLess{}, s));
    DPHY_CUDA(ctx, cub::DeviceReduce::ReduceByKey(nullptr, rbk_bytes, (const CladeKey*)nullptr, (CladeKey*)nullptr, (const CladeVal*)nullptr,
                                                  (CladeVal*)nullptr, (int32_t*)nullptr, CladeValAdd{}, m, s));
    Slab mg;
    const int b_mkey = mg.reserve(sizeof(CladeKey) * (size_t)m), b_mval = mg.reserve(sizeof(CladeVal) * (size_t)m);
    const int b_mcub = mg.reserve(std::max(merge_bytes, rbk_bytes));
    DevBlock mblk(s);
    if (!mblk.alloc(mg.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(clade table merge)");
    CladeKey* mkey = mg.at<CladeKey>(mblk.p, b_mkey);
    CladeVal* mval = mg.at<CladeVal>(mblk.p, b_mval);
    void* mcub = mg.at<char>(mblk.p, b_mcub);
    DPHY_CUDA(ctx, cub::DeviceMerge::MergePairs(mcub, merge_bytes, (const CladeKey*)tab->d_keys, (const CladeVal*)tab->d_vals, (int)nt,
                                                (const CladeKey*)bkey, (const CladeVal*)bval, nb, mkey, mval, CladeKeyLess{}, s));
    DPHY_CUDA(ctx, cub::DeviceReduce::ReduceByKey(mcub, rbk_bytes, (const CladeKey*)mkey, new_keys, (const CladeVal*)mval, new_vals, d_nruns,
                                                  CladeValAdd{}, m, s));
    ctx->launches += 4;
    DPHY_CUDA(ctx, cudaMemcpyAsync(&n_out, d_nruns, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  }
  DPHY_CUDA(ctx, cudaStreamSynchronize(s));
  if (n_out != n_new) return set_error(ctx, DPHY_ERR_INTERNAL, "clade table: merged clade count disagrees with the lookup");

  // ---- step 4: commit
  if (tab->d_keys) cudaFreeAsync(tab->d_keys, s);
  tab->d_keys = new_keys;
  tab->d_vals = new_vals;
  table_blk.release();
  if (first) {
    tab->d_tips = (uint32_t*)tips_blk.release();
    tab->num_nodes = Nt;
    tab->num_tips = (int32_t)tips_per_tree;
  }
  tab->num_trees += T;
  tab->num_clades = n_new;
  tab->bytes = sizeof(uint32_t) * (size_t)words + (sizeof(CladeKey) + sizeof(CladeVal)) * (size_t)n_new;
  return DPHY_OK;
}

int dphy_clade_table_score(dphy_ctx* ctx, dphy_clade_table* tab, dphy_forest* fo, double* out) {
  int st = check_use(ctx, tab, fo);
  if (st != DPHY_OK) return st;
  if (!out) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "clade table score: out is NULL");
  if (tab->num_trees == 0) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "clade table score: no tree has been added");
  const int T = fo->h.num_trees, tiles = fo->h.num_tiles;
  if (T == 0) return DPHY_OK;
  int Nt;
  if ((st = check_sizes(ctx, tab, fo, &Nt)) != DPHY_OK) return st;
  cudaSetDevice(ctx->device);
  KeyScratch ks(ctx->stream);
  Slab ex;
  const int b_part = ex.reserve(sizeof(double) * tiles), b_out = ex.reserve(sizeof(double) * T);
  if ((st = clade_keys(ctx, fo, tab->d_tips, 0, ex.total, ks)) != DPHY_OK) return st;
  double* tile_part = ex.at<double>(ks.extra, b_part);
  double* d_out = ex.at<double>(ks.extra, b_out);
  clade_score_tile_kernel<<<tiles, kTile, 0, ctx->stream>>>(fo->h, ks.h, view_of(tab), tile_part);
  clade_tree_sum_kernel<<<T, kTile, 0, ctx->stream>>>(fo->h, tile_part, d_out);
  ctx->launches += 2;
  DPHY_CUDA(ctx, cudaGetLastError());
  unsigned long long hst[kStLen];
  std::vector<double> h_out(T);
  DPHY_CUDA(ctx, cudaMemcpyAsync(hst, ks.status, sizeof(hst), cudaMemcpyDeviceToHost, ctx->stream));
  DPHY_CUDA(ctx, cudaMemcpyAsync(h_out.data(), d_out, sizeof(double) * T, cudaMemcpyDeviceToHost, ctx->stream));
  DPHY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (!tips_ok(hst, T, tab->num_tips))
    return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "clade table score: every tree must have the same tips (host node indices) as the table's");
  std::memcpy(out, h_out.data(), sizeof(double) * T);
  return DPHY_OK;
}

int dphy_clade_table_node_support(dphy_ctx* ctx, dphy_clade_table* tab, dphy_forest* fo, int32_t tree, int64_t* count, double* mean_t) {
  int st = check_use(ctx, tab, fo);
  if (st != DPHY_OK) return st;
  if (!count || !mean_t) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "clade table node support: count and mean_t are required");
  if (tree < 0 || tree >= fo->h.num_trees) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "clade table node support: tree index out of range");
  if (tab->num_trees == 0) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "clade table node support: no tree has been added");
  int Nt;
  if ((st = check_sizes(ctx, tab, fo, &Nt)) != DPHY_OK) return st;
  cudaSetDevice(ctx->device);
  KeyScratch ks(ctx->stream);
  Slab ex;
  const int b_count = ex.reserve(sizeof(int64_t) * Nt), b_mean = ex.reserve(sizeof(double) * Nt);
  if ((st = clade_keys(ctx, fo, tab->d_tips, 0, ex.total, ks)) != DPHY_OK) return st;
  int64_t* d_count = ex.at<int64_t>(ks.extra, b_count);
  double* d_mean = ex.at<double>(ks.extra, b_mean);
  clade_node_support_kernel<<<blocks(Nt), 256, 0, ctx->stream>>>(fo->h, tree, ks.h, view_of(tab), d_count, d_mean);
  ++ctx->launches;
  DPHY_CUDA(ctx, cudaGetLastError());
  unsigned long long hst[kStLen];
  std::vector<int64_t> h_count(Nt);
  std::vector<double> h_mean(Nt);
  DPHY_CUDA(ctx, cudaMemcpyAsync(hst, ks.status, sizeof(hst), cudaMemcpyDeviceToHost, ctx->stream));
  DPHY_CUDA(ctx, cudaMemcpyAsync(h_count.data(), d_count, sizeof(int64_t) * Nt, cudaMemcpyDeviceToHost, ctx->stream));
  DPHY_CUDA(ctx, cudaMemcpyAsync(h_mean.data(), d_mean, sizeof(double) * Nt, cudaMemcpyDeviceToHost, ctx->stream));
  DPHY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (!tips_ok(hst, fo->h.num_trees, tab->num_tips))
    return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "clade table node support: every tree must have the same tips (host node indices) as the table's");
  std::memcpy(count, h_count.data(), sizeof(int64_t) * Nt);
  std::memcpy(mean_t, h_mean.data(), sizeof(double) * Nt);
  return DPHY_OK;
}

}  // extern "C"
