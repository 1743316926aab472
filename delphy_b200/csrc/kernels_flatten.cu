// kernels_flatten.cu -- device-side flattening of host-order EMATs into the forest layout (sm_100a).
//
// The reference keeps a Phylo_tree as an index-based AoS binary tree (core/tree.h:181-220, core/phylo_tree.h:14-63);
// the C ABI receives it as SoA + CSR arrays in HOST node order.  Every kernel of the hot path wants DFS pre-order
// (children[1] first -- the order of Spr_study_builder's LIFO work stack, core/spr_study.cpp:103-128).  Doing that
// re-ordering on the host costs a sequential, cache-hostile DFS per upload and dominated the end-to-end time, so the
// host now only streams the raw arrays to the device and the re-ordering happens here:
//
//   1. Euler tour: every node gets an "enter" and an "exit" arc; succ(enter v) = enter(child1 v) or exit(v) for a tip;
//      succ(exit v) = enter(child0 of parent) if v is children[1], exit(parent) if v is children[0], end for the root.
//   2. Wyllie list ranking (pointer jumping, ceil(log2(2N)) rounds, ping-pong buffers) carrying two suffix counters:
//      E = #enter arcs and A = #arcs from here to the end of the tour.  Then
//         pre-order index  = N - E[enter v]            subtree size = E[enter v] - E[exit v]
//         depth            = 2 pre - (2N - A[enter v]) post-order index = (2N - A[exit v]) - (N - E[exit v])
//   3. scatter node records to device order, exclusive-scan the per-node list lengths into the device CSR offsets,
//      gather the mutation / missation / from-state lists (packing partition|from|to codes, validating ranges).
//
// All validation the reference performs by CHECK / std::out_of_range (core/mutations.h:187-191, core/phylo_tree.cpp:18-135
// for the topology part) is folded into these kernels and reported through one status word.
#include "dphy_internal.h"
#include "device_utils.cuh"

#include <algorithm>

namespace dphy {

constexpr int kScanItems = 4;                       // items per thread in the offset scans
constexpr int kScanTile = kTile * kScanItems;       // 1024 positions per scan tile

__device__ __forceinline__ void flag_error(FlattenParams& P, uint32_t bit) { atomicOr(P.status, bit); }

// ---- (1) Euler-tour arcs + topology validation ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(kTile) flatten_arcs_init_kernel(FlattenParams P) {
  const int tile = blockIdx.x;
  const int tree = P.tile_tree[tile];
  const TreeDev T = P.trees[tree];
  const RawTreeDev R = P.raw[tree];
  const int v = (tile - T.first_tile) * kTile + threadIdx.x;
  if (v >= T.num_nodes) return;
  const int n = T.num_nodes;
  const int g = T.node_base + v;
  const int par = R.parent[v], c0 = R.child0[v], c1 = R.child1[v];
  bool ok = true;
  const bool is_root = (v == R.root);
  const bool internal = (c0 >= 0 || c1 >= 0);
  if (internal) {
    ok = c0 >= 0 && c1 >= 0 && c0 < n && c1 < n && c0 != c1 && c0 != v && c1 != v;
    if (ok) ok = R.parent[c0] == v && R.parent[c1] == v;
  }
  if (is_root) ok = ok && par == -1;
  else {
    ok = ok && par >= 0 && par < n && par != v;
    if (ok) ok = (R.child0[par] == v) != (R.child1[par] == v);
  }
  int succ_enter, succ_exit;
  if (!ok) {
    flag_error(P, kFlattenErrTopology);
    succ_enter = 2 * g + 1; succ_exit = -1;          // harmless self-contained list
  } else {
    succ_enter = internal ? 2 * (T.node_base + c1) : 2 * g + 1;
    if (is_root) succ_exit = -1;
    else if (R.child1[par] == v) succ_exit = 2 * (T.node_base + R.child0[par]);
    else succ_exit = 2 * (T.node_base + par) + 1;
  }
  P.arcs[0][2 * g] = make_int4(succ_enter, 1, 1, 0);
  P.arcs[0][2 * g + 1] = make_int4(succ_exit, 0, 1, 0);
}

// ---- (2) one pointer-jumping round -----------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) flatten_rank_round_kernel(const int4* __restrict__ src, int4* __restrict__ dst, int num_arcs) {
  const int a = blockIdx.x * 256 + threadIdx.x;
  if (a >= num_arcs) return;
  int4 x = src[a];
  if (x.x >= 0) {
    const int4 y = __ldg(src + x.x);
    x.x = y.x; x.y += y.y; x.z += y.z;
  }
  dst[a] = x;
}

// ---- (3a) node records to device order; per-node list lengths ----------------------------------------------------------------------------
__global__ void __launch_bounds__(kTile) flatten_nodes_kernel(FlattenParams P, int final_buf) {
  const int tile = blockIdx.x;
  const int tree = P.tile_tree[tile];
  const TreeDev T = P.trees[tree];
  const RawTreeDev R = P.raw[tree];
  const int v = (tile - T.first_tile) * kTile + threadIdx.x;
  if (v >= T.num_nodes) return;
  const int n = T.num_nodes;
  const int g = T.node_base + v;
  const int4* arcs = P.arcs[final_buf];
  const int4 en = arcs[2 * g], ex = arcs[2 * g + 1];
  const int pre = n - en.y;
  const int pos_a = 2 * n - en.z;
  const int depth = 2 * pre - pos_a;
  const int size = en.y - ex.y;
  const int post = (2 * n - ex.z) - (n - ex.y);
  bool ok = en.x < 0 && ex.x < 0 && pre >= 0 && pre < n && size >= 1 && pre + size <= n && post >= 0 && post < n && depth >= 0;
  if (v == R.root) ok = ok && en.y == n && en.z == 2 * n;     // every node is reachable from the root
  if (!ok) { flag_error(P, kFlattenErrTopology); return; }
  const int p = T.node_base + pre;
  P.node_id[p] = v;
  P.pos_of_node[g] = pre;
  P.depth[p] = depth;
  P.subtree_size[p] = size;
  P.t[p] = R.t[v];
  P.post_node[T.node_base + post] = p;
  const int par = R.parent[v];
  P.parent_pos[p] = par < 0 ? -1 : T.node_base + (n - arcs[2 * (T.node_base + par)].y);
  // times never decrease away from the root (core/phylo_tree.cpp:131): the SPR kernels prune whole subtrees on that invariant
  if (par >= 0 && R.t[v] < R.t[par]) flag_error(P, kFlattenErrTimes);
  int cm = R.mut_off[v + 1] - R.mut_off[v], ci = R.miss_off[v + 1] - R.miss_off[v], cf = R.fs_off[v + 1] - R.fs_off[v];
  if (cm < 0 || ci < 0 || cf < 0 || R.mut_off[v] < 0 || R.miss_off[v] < 0 || R.fs_off[v] < 0 ||
      R.mut_off[v + 1] > R.num_muts || R.miss_off[v + 1] > R.num_ivls || R.fs_off[v + 1] > R.num_fs) {
    flag_error(P, kFlattenErrOffsets); cm = ci = cf = 0;
  }
  P.mut_off[p] = cm; P.miss_off[p] = ci; P.fs_off[p] = cf;
  atomicMax(P.max_depth + tree, depth);
  // straddler: closes (is subtracted from the running lambda) at position pre+size, which lies in a later log-G tile
  if (pre + size < n && pre / kLgTile != (pre + size) / kLgTile) {
    const uint32_t slot = atomicAdd(P.status + 1, 1u);
    P.strad_list[2 * slot] = p; P.strad_list[2 * slot + 1] = T.sites_id;
  }
}

// ---- (3b) exclusive scan of the three length arrays, in place, over the whole forest ------------------------------------------------------------
__global__ void __launch_bounds__(kTile) flatten_scan_reduce_kernel(FlattenParams P) {
  __shared__ int s_ws[kTile / 32];
  const int base = blockIdx.x * kScanTile;
  int a = 0, b = 0, c = 0;
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) {
    const int i = base + k * kTile + threadIdx.x;
    if (i < P.num_nodes) { a += P.mut_off[i]; b += P.miss_off[i]; c += P.fs_off[i]; }
  }
  a = block_sum<int, kTile>(a, s_ws);
  b = block_sum<int, kTile>(b, s_ws);
  c = block_sum<int, kTile>(c, s_ws);
  if (threadIdx.x == 0) { P.scan_tiles[blockIdx.x * 3 + 0] = a; P.scan_tiles[blockIdx.x * 3 + 1] = b; P.scan_tiles[blockIdx.x * 3 + 2] = c; }
}

__global__ void __launch_bounds__(1024) flatten_scan_spine_kernel(FlattenParams P, int num_scan_tiles) {
  __shared__ int s_ws[32];
  __shared__ int s_carry[3];
  if (threadIdx.x < 3) s_carry[threadIdx.x] = 0;
  __syncthreads();
  for (int j0 = 0; j0 < num_scan_tiles; j0 += 1024) {
    const int j = j0 + threadIdx.x;
    const bool ok = j < num_scan_tiles;
    int tot[3];
#pragma unroll
    for (int w = 0; w < 3; ++w) {
      const int v = ok ? P.scan_tiles[j * 3 + w] : 0;
      const int incl = block_scan_incl<int, 1024>(v, s_ws, &tot[w]);
      if (ok) P.scan_tiles[j * 3 + w] = s_carry[w] + incl - v;
      __syncthreads();
    }
    if (threadIdx.x < 3) s_carry[threadIdx.x] += tot[threadIdx.x];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    P.mut_off[P.num_nodes] = s_carry[0]; P.miss_off[P.num_nodes] = s_carry[1]; P.fs_off[P.num_nodes] = s_carry[2];
    if (s_carry[0] != P.total_muts || s_carry[1] != P.total_ivls || s_carry[2] != P.total_fs) atomicOr(P.status, kFlattenErrOffsets);
  }
}

__global__ void __launch_bounds__(kTile) flatten_scan_apply_kernel(FlattenParams P) {
  __shared__ int s_ws[kTile / 32];
  const int base = blockIdx.x * kScanTile + threadIdx.x * kScanItems;
  int32_t* arrs[3] = {P.mut_off, P.miss_off, P.fs_off};
#pragma unroll
  for (int w = 0; w < 3; ++w) {
    int v[kScanItems], run = 0;
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) { v[k] = base + k < P.num_nodes ? arrs[w][base + k] : 0; run += v[k]; }
    int tot;
    const int incl = block_scan_incl<int, kTile>(run, s_ws, &tot);
    int ex = P.scan_tiles[blockIdx.x * 3 + w] + incl - run;
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) { if (base + k < P.num_nodes) arrs[w][base + k] = ex; ex += v[k]; }
    __syncthreads();
  }
}

// ---- (3c) lists to device order: packed codes + range validation -------------------------------------------------------------------------
// One CTA per tile of kTile device positions.  The destination ranges of a tile are contiguous (CSR in device order), so the
// lists are copied FLAT -- one destination event per thread, its node found by binary search in the tile's offsets held in
// shared memory -- which keeps every store coalesced and the gathers independent, however the events spread over the nodes.
__device__ __forceinline__ int tile_owner(const int* s_dst, int e) {   // last n in [0, kTile) with s_dst[n] <= e
  int lo = 0, hi = kTile - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (s_dst[mid] <= e) lo = mid; else hi = mid - 1;
  }
  return lo;
}

__global__ void __launch_bounds__(kTile) flatten_events_kernel(FlattenParams P) {
  __shared__ int s_dst[3][kTile + 1];
  __shared__ int s_src[3][kTile];
  const int tile = blockIdx.x + P.tile_base, tid = threadIdx.x;
  const int tree = P.tile_tree[tile];
  const TreeDev T = P.trees[tree];
  const RawTreeDev R = P.raw[tree];
  const SitesDev& S = P.sites[T.sites_id];
  const int q0 = (tile - T.first_tile) * kTile;
  const int n_act = min(kTile, T.num_nodes - q0);
  const int p0 = T.node_base + q0;
  const int L = S.L;
  {
    const int p = p0 + min(tid, n_act);          // inactive threads repeat the end offsets: they own no event
    const int v = tid < n_act ? P.node_id[p] : 0;
    s_dst[0][tid] = P.mut_off[p]; s_dst[1][tid] = P.miss_off[p]; s_dst[2][tid] = P.fs_off[p];
    s_src[0][tid] = tid < n_act ? R.mut_off[v] : 0; s_src[1][tid] = tid < n_act ? R.miss_off[v] : 0; s_src[2][tid] = tid < n_act ? R.fs_off[v] : 0;
    if (tid == 0) { s_dst[0][kTile] = P.mut_off[p0 + n_act]; s_dst[1][kTile] = P.miss_off[p0 + n_act]; s_dst[2][kTile] = P.fs_off[p0 + n_act]; }
  }
  __syncthreads();
  uint32_t err = 0;
  for (int e = s_dst[0][0] + tid; e < s_dst[0][kTile]; e += kTile) {
    const int n = tile_owner(s_dst[0], e);
    const int src = s_src[0][n] + (e - s_dst[0][n]);
    int l = R.mut_site[src];
    const int from = R.mut_from[src], to = R.mut_to[src];
    if (l < 0 || l >= L) { err |= kFlattenErrMutSite; l = 0; }
    if (from > 3 || to > 3) err |= kFlattenErrMutState;
    P.mut_site[e] = l;
    P.mut_code[e] = (uint8_t)(S.part[l] << 4 | (from & 3) << 2 | (to & 3));
    P.mut_t[e] = R.mut_t[src];
  }
  for (int e = s_dst[1][0] + tid; e < s_dst[1][kTile]; e += kTile) {
    const int n = tile_owner(s_dst[1], e);
    const int src = s_src[1][n] + (e - s_dst[1][n]);
    int s0 = R.miss_start[src], s1 = R.miss_end[src];
    if (s0 < 0 || s1 > L || s0 >= s1) { err |= kFlattenErrMissation; s0 = 0; s1 = 1; }   // core/mutations.h:187-191
    P.miss_se[e] = make_int2(s0, s1);
  }
  for (int e = s_dst[2][0] + tid; e < s_dst[2][kTile]; e += kTile) {
    const int n = tile_owner(s_dst[2], e);
    const int src = s_src[2][n] + (e - s_dst[2][n]);
    int l = R.fs_site[src];
    const int from = R.fs_from[src];
    if (l < 0 || l >= L) { err |= kFlattenErrMissation; l = 0; }
    if (from > 3) err |= kFlattenErrFsState;
    P.fs_site[e] = l;
    P.fs_code[e] = (uint8_t)(S.part[l] << 4 | S.ref[l] << 2 | (from & 3));
  }
  if (err) flag_error(P, err);
}

// ---- (3d) every per-branch list folded into one 4P-vector of state counts (see ForestDev::bw; fsw = the from-state part) -----------
// Structure only: depends on the tree, its lists, the reference sequence and the partition map -- not on the evo model.
// Flat over the tile's events again; an interval turns into 4P counts with two 16-byte look-ups per partition in the
// interleaved cumulative table cref[l][4P]; per-node sums are integer shared-memory atomics (exact, order-free).
constexpr int kBwRow = kMaxPartitions * 4 + 1;      // padded row: conflict-free when every thread walks its own row
__global__ void __launch_bounds__(kTile) fold_branch_weights_kernel(FlattenParams P) {
  __shared__ int s_w[kTile * kBwRow];
  __shared__ int s_f[kTile * kBwRow];
  __shared__ int s_dst[3][kTile + 1];
  const int tile = blockIdx.x + P.tile_base, tid = threadIdx.x;
  const int tree = P.tile_tree[tile];
  const TreeDev T = P.trees[tree];
  const SitesDev& S = P.sites[T.sites_id];
  const int q0 = (tile - T.first_tile) * kTile;
  const int n_act = min(kTile, T.num_nodes - q0);
  const int p0 = T.node_base + q0;
  const int stride = P.fsw_stride, K = S.P * 4;
  for (int i = tid; i < kTile * kBwRow; i += kTile) { s_w[i] = 0; s_f[i] = 0; }
  {
    const int p = p0 + min(tid, n_act);
    s_dst[0][tid] = P.mut_off[p]; s_dst[1][tid] = P.miss_off[p]; s_dst[2][tid] = P.fs_off[p];
    if (tid == 0) { s_dst[0][kTile] = P.mut_off[p0 + n_act]; s_dst[1][kTile] = P.miss_off[p0 + n_act]; s_dst[2][kTile] = P.fs_off[p0 + n_act]; }
  }
  __syncthreads();
  for (int e = s_dst[0][0] + tid; e < s_dst[0][kTile]; e += kTile) {
    const int n = tile_owner(s_dst[0], e);
    const int code = P.mut_code[e], pt = code >> 4, x = (code >> 2) & 3, y = code & 3;
    if (x != y) { atomicAdd(&s_w[n * kBwRow + pt * 4 + y], 1); atomicSub(&s_w[n * kBwRow + pt * 4 + x], 1); }
  }
  const int4* __restrict__ cref4 = reinterpret_cast<const int4*>(S.cref);
  for (int e = s_dst[1][0] + tid; e < s_dst[1][kTile]; e += kTile) {
    const int n = tile_owner(s_dst[1], e);
    const int2 se = P.miss_se[e];
    for (int b = 0; b < S.P; ++b) {
      const int4 hi = __ldg(cref4 + (size_t)se.y * S.P + b), lo = __ldg(cref4 + (size_t)se.x * S.P + b);
      int* w = &s_w[n * kBwRow + b * 4];
      if (hi.x != lo.x) atomicSub(w + 0, hi.x - lo.x);
      if (hi.y != lo.y) atomicSub(w + 1, hi.y - lo.y);
      if (hi.z != lo.z) atomicSub(w + 2, hi.z - lo.z);
      if (hi.w != lo.w) atomicSub(w + 3, hi.w - lo.w);
    }
  }
  for (int e = s_dst[2][0] + tid; e < s_dst[2][kTile]; e += kTile) {
    const int n = tile_owner(s_dst[2], e);
    const int code = P.fs_code[e], pt = code >> 4, rf = (code >> 2) & 3, fr = code & 3;
    if (rf != fr) { atomicAdd(&s_f[n * kBwRow + pt * 4 + rf], 1); atomicSub(&s_f[n * kBwRow + pt * 4 + fr], 1); }
  }
  __syncthreads();
  if (tid < n_act) {
    const int p = p0 + tid;
    for (int k = 0; k < stride; ++k) {
      const int fk = k < K ? s_f[tid * kBwRow + k] : 0;
      if (fk > 32767 || fk < -32768) flag_error(P, kFlattenErrFswRange);
      P.fsw[(size_t)p * stride + k] = (int16_t)fk;
      P.C[(size_t)p * stride + k] = (k < K ? s_w[tid * kBwRow + k] : 0) + fk;   // bw; turned into C by the count scan below
    }
  }
}

// ---- (3e) per-node state counts: C[q] = sum of bw over the root -> q path (see ForestDev::C) ---------------------------------------------
// With X the inclusive prefix of bw over the forest in device order and Y the exclusive prefix of bw over the post-order lists
// (tree after tree), C[q] = X[q] - Y[q - depth[q]]: the nodes opened up to q minus the q - depth[q] nodes of q's tree closed before
// q.  Every tree's post-order list holds exactly that tree's nodes, so the earlier trees' totals cancel.  X and Y may wrap; they
// are summed as uint32, and the difference, a bounded state count, comes out exact.  Each int4 column group of the rows is
// scanned on its own (blockIdx.y); bw lies in P.C, and the last kernel replaces it in place.
__device__ __forceinline__ uint4 u4_add(uint4 a, uint4 b) { return make_uint4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ uint4 u4_sub(uint4 a, uint4 b) { return make_uint4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w); }
__device__ __forceinline__ uint4 u4_shfl_up(uint4 v, int o) {
  return make_uint4(__shfl_up_sync(0xffffffffu, v.x, o), __shfl_up_sync(0xffffffffu, v.y, o), __shfl_up_sync(0xffffffffu, v.z, o),
                    __shfl_up_sync(0xffffffffu, v.w, o));
}
// inclusive block scan of one uint4 per thread (blockDim.x == kTile); *total = the block total
__device__ __forceinline__ uint4 block_scan_incl_u4(uint4 v, uint4* ws, uint4* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint4 u = u4_shfl_up(v, o);
    if (lane >= o) v = u4_add(v, u);
  }
  if (lane == 31) ws[warp] = v;
  __syncthreads();
  uint4 base = make_uint4(0, 0, 0, 0), tot = make_uint4(0, 0, 0, 0);
#pragma unroll
  for (int w = 0; w < kTile / 32; ++w) { if (w < warp) base = u4_add(base, ws[w]); tot = u4_add(tot, ws[w]); }
  __syncthreads();                         // ws may be rewritten by the next scan
  *total = tot;
  return u4_add(base, v);
}

// per scan tile of kScanTile rows: totals of X's and Y's terms -> cnt_tot[(tile * G + g) * 2 + {0, 1}]
__global__ void __launch_bounds__(kTile) counts_scan_reduce_kernel(FlattenParams P) {
  __shared__ uint4 s_ws[kTile / 32];
  const int G = P.fsw_stride / 4, g = blockIdx.y;
  const uint4* __restrict__ bw4 = reinterpret_cast<const uint4*>(P.C);
  const int base = blockIdx.x * kScanTile + threadIdx.x * kScanItems;
  uint4 a = make_uint4(0, 0, 0, 0), b = make_uint4(0, 0, 0, 0);
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) {
    const int i = base + k;
    if (i < P.num_nodes) {
      a = u4_add(a, bw4[(size_t)i * G + g]);
      b = u4_add(b, bw4[(size_t)P.post_node[i] * G + g]);
    }
  }
  uint4 ta, tb;
  block_scan_incl_u4(a, s_ws, &ta);
  block_scan_incl_u4(b, s_ws, &tb);
  if (threadIdx.x == 0) {
    P.cnt_tot[((size_t)blockIdx.x * G + g) * 2 + 0] = ta;
    P.cnt_tot[((size_t)blockIdx.x * G + g) * 2 + 1] = tb;
  }
}

// exclusive prefix of the tile totals, in place: one CTA per (column group, X | Y)
__global__ void __launch_bounds__(kTile) counts_scan_spine_kernel(FlattenParams P, int num_scan_tiles) {
  __shared__ uint4 s_ws[kTile / 32];
  const int G = P.fsw_stride / 4, col = blockIdx.x;            // col = g * 2 + (0: X, 1: Y)
  uint4 carry = make_uint4(0, 0, 0, 0);
  for (int j0 = 0; j0 < num_scan_tiles; j0 += kTile) {
    const int j = j0 + threadIdx.x;
    uint4* slot = P.cnt_tot + ((size_t)j * G) * 2 + col;
    const uint4 v = j < num_scan_tiles ? *slot : make_uint4(0, 0, 0, 0);
    uint4 tot;
    const uint4 incl = block_scan_incl_u4(v, s_ws, &tot);
    if (j < num_scan_tiles) *slot = u4_add(carry, u4_sub(incl, v));
    carry = u4_add(carry, tot);
  }
}

// Y: exclusive prefix of bw over the post-order lists -> cnt_y
__global__ void __launch_bounds__(kTile) counts_scan_post_kernel(FlattenParams P) {
  __shared__ uint4 s_ws[kTile / 32];
  const int G = P.fsw_stride / 4, g = blockIdx.y;
  const uint4* __restrict__ bw4 = reinterpret_cast<const uint4*>(P.C);
  uint4* __restrict__ y4 = reinterpret_cast<uint4*>(P.cnt_y);
  const int base = blockIdx.x * kScanTile + threadIdx.x * kScanItems;
  uint4 v[kScanItems], run = make_uint4(0, 0, 0, 0);
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) {
    v[k] = base + k < P.num_nodes ? bw4[(size_t)P.post_node[base + k] * G + g] : make_uint4(0, 0, 0, 0);
    run = u4_add(run, v[k]);
  }
  uint4 tot;
  uint4 ex = u4_sub(block_scan_incl_u4(run, s_ws, &tot), run);
  ex = u4_add(ex, P.cnt_tot[((size_t)blockIdx.x * G + g) * 2 + 1]);
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) { if (base + k < P.num_nodes) y4[(size_t)(base + k) * G + g] = ex; ex = u4_add(ex, v[k]); }
}

// C[q] = X[q] - Y[q - depth[q]], X formed here (inclusive prefix of bw in device order), written over bw in place
__global__ void __launch_bounds__(kTile) counts_scan_apply_kernel(FlattenParams P) {
  __shared__ uint4 s_ws[kTile / 32];
  const int G = P.fsw_stride / 4, g = blockIdx.y;
  uint4* __restrict__ c4 = reinterpret_cast<uint4*>(P.C);
  const uint4* __restrict__ y4 = reinterpret_cast<const uint4*>(P.cnt_y);
  const int base = blockIdx.x * kScanTile + threadIdx.x * kScanItems;
  uint4 v[kScanItems], run = make_uint4(0, 0, 0, 0);
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) {
    v[k] = base + k < P.num_nodes ? c4[(size_t)(base + k) * G + g] : make_uint4(0, 0, 0, 0);
    run = u4_add(run, v[k]);
  }
  uint4 tot;
  uint4 x = u4_sub(block_scan_incl_u4(run, s_ws, &tot), run);
  x = u4_add(x, P.cnt_tot[((size_t)blockIdx.x * G + g) * 2 + 0]);
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) {
    const int q = base + k;
    x = u4_add(x, v[k]);
    if (q < P.num_nodes) c4[(size_t)q * G + g] = u4_sub(x, y4[(size_t)(q - P.depth[q]) * G + g]);
  }
}

// ---- (4) log-G tile descriptors: the tile's slice of the tree's post-order list ----------------------------------------------
__global__ void __launch_bounds__(256) flatten_ctiles_kernel(FlattenParams P) {
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j >= P.num_ctiles) return;
  CTileDesc& d = P.ctiles[j];
  const int p0 = d.tile_start, p1 = d.tile_start + d.n_act;
  const int q_first = p0 - d.node_base, q_last = p1 - 1 - d.node_base;
  d.cl0 = q_first == 0 ? 0 : (q_first - 1) - P.depth[p0 - 1];
  d.cl1 = q_last - P.depth[p1 - 1];
}

// Accepted displace moves (core/subrun.cpp:223-231,276-284): scatter new node times by host node index.
__global__ void set_node_times_kernel(const int32_t* __restrict__ pos_of_node, double* __restrict__ t, int node_base, int num_nodes,
                                      const int32_t* __restrict__ nodes, const double* __restrict__ vals, int count, uint32_t* status) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const int v = nodes[i];
  if (v < 0 || v >= num_nodes) { atomicOr(status, 1u); return; }
  t[node_base + pos_of_node[node_base + v]] = vals[i];
}

// After the scatter: every displaced node must still lie between its parent and its children (status bit 1).
__global__ void check_node_times_kernel(const int32_t* __restrict__ pos_of_node, const double* __restrict__ t, const int32_t* __restrict__ parent_pos,
                                        const int32_t* __restrict__ subtree_size, int node_base, int num_nodes,
                                        const int32_t* __restrict__ nodes, int count, uint32_t* status) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const int v = nodes[i];
  if (v < 0 || v >= num_nodes) return;
  const int p = node_base + pos_of_node[node_base + v];
  const int par = parent_pos[p];
  bool bad = par >= 0 && t[p] < t[par];
  if (subtree_size[p] > 1) {
    const int c1 = p + 1, c0 = p + 1 + subtree_size[p + 1];
    bad = bad || t[c1] < t[p] || t[c0] < t[p];
  }
  if (bad) atomicOr(status, 2u);
}

int launch_set_node_times(dphy_ctx* ctx, dphy_forest* fo, int tree, const int32_t* d_nodes, const double* d_vals, int count, uint32_t* d_status) {
  const TreeDev& T = fo->trees[tree];
  set_node_times_kernel<<<(count + 255) / 256, 256, 0, ctx->stream>>>(fo->h.pos_of_node, fo->h.t, T.node_base, T.num_nodes, d_nodes, d_vals, count, d_status);
  check_node_times_kernel<<<(count + 255) / 256, 256, 0, ctx->stream>>>(fo->h.pos_of_node, fo->h.t, fo->h.parent_pos, fo->h.subtree_size,
                                                                        T.node_base, T.num_nodes, d_nodes, count, d_status);
  ctx->launches += 2;
  return check_cuda(ctx, cudaGetLastError(), "set_node_times_kernel");
}

// The node records of trees whose links are those of the forest being replaced: same DFS order, depth and subtree sizes (copied through
// the old position of every node), fresh times and list lengths, the same checks as flatten_nodes_kernel.
__global__ void __launch_bounds__(kTile) flatten_nodes_reuse_kernel(FlattenParams P) {
  const int tile = blockIdx.x;
  const int tree = P.tile_tree[tile];
  const TreeDev T = P.trees[tree];
  const RawTreeDev R = P.raw[tree];
  const int v = (tile - T.first_tile) * kTile + threadIdx.x;
  if (v >= T.num_nodes) return;
  const int n = T.num_nodes;
  const int g = T.node_base + v;
  const int pre = P.old_pos_of_node[g];
  const int p = T.node_base + pre;
  const int depth = P.old_depth[p], size = P.old_subtree_size[p];
  P.node_id[p] = v;
  P.pos_of_node[g] = pre;
  P.depth[p] = depth;
  P.subtree_size[p] = size;
  P.t[p] = R.t[v];
  P.post_node[T.node_base + pre + size - 1 - depth] = p;        // post-order index of a node = pre + size - 1 - depth
  const int par = R.parent[v];
  P.parent_pos[p] = P.old_parent_pos[p];
  if (par >= 0 && R.t[v] < R.t[par]) flag_error(P, kFlattenErrTimes);
  int cm = R.mut_off[v + 1] - R.mut_off[v], ci = R.miss_off[v + 1] - R.miss_off[v], cf = R.fs_off[v + 1] - R.fs_off[v];
  if (cm < 0 || ci < 0 || cf < 0 || R.mut_off[v] < 0 || R.miss_off[v] < 0 || R.fs_off[v] < 0 ||
      R.mut_off[v + 1] > R.num_muts || R.miss_off[v + 1] > R.num_ivls || R.fs_off[v + 1] > R.num_fs) {
    flag_error(P, kFlattenErrOffsets); cm = ci = cf = 0;
  }
  P.mut_off[p] = cm; P.miss_off[p] = ci; P.fs_off[p] = cf;
  atomicMax(P.max_depth + tree, depth);
  if (pre + size < n && pre / kLgTile != (pre + size) / kLgTile) {
    const uint32_t slot = atomicAdd(P.status + 1, 1u);
    P.strad_list[2 * slot] = p; P.strad_list[2 * slot + 1] = T.sites_id;
  }
}

int launch_flatten(dphy_ctx* ctx, const FlattenParams& P, int num_tiles, int max_tree_nodes, int stage) {
  if (P.num_nodes == 0) return DPHY_OK;
  const int num_arcs = 2 * P.num_nodes;
  int rounds = 0;
  while ((1LL << rounds) < 2LL * max_tree_nodes) ++rounds;
  const bool reuse = P.old_pos_of_node != nullptr;
  if (reuse && stage == 0) return DPHY_OK;       // nothing to rank
  if ((stage < 0 || stage == 0) && !reuse) {
    flatten_arcs_init_kernel<<<num_tiles, kTile, 0, ctx->stream>>>(P);
    for (int r = 0; r < rounds; ++r)
      flatten_rank_round_kernel<<<(num_arcs + 255) / 256, 256, 0, ctx->stream>>>(P.arcs[r & 1], P.arcs[(r + 1) & 1], num_arcs);
    ctx->launches += 1 + rounds;
    if (stage == 0) return check_cuda(ctx, cudaGetLastError(), "flatten kernels launch (topology)");
  }
  if (stage < 0 || stage == 1) {
    if (reuse) flatten_nodes_reuse_kernel<<<num_tiles, kTile, 0, ctx->stream>>>(P);
    else flatten_nodes_kernel<<<num_tiles, kTile, 0, ctx->stream>>>(P, rounds & 1);
    const int nst = (P.num_nodes + kScanTile - 1) / kScanTile;
    flatten_scan_reduce_kernel<<<nst, kTile, 0, ctx->stream>>>(P);
    flatten_scan_spine_kernel<<<1, 1024, 0, ctx->stream>>>(P, nst);
    flatten_scan_apply_kernel<<<nst, kTile, 0, ctx->stream>>>(P);
    ctx->launches += 4;
    if (stage == 1) return check_cuda(ctx, cudaGetLastError(), "flatten kernels launch (node records)");
  }
  flatten_events_kernel<<<num_tiles, kTile, 0, ctx->stream>>>(P);
  fold_branch_weights_kernel<<<num_tiles, kTile, 0, ctx->stream>>>(P);
  ctx->launches += 2;
  const int st = check_cuda(ctx, cudaGetLastError(), "flatten kernels launch");
  return st != DPHY_OK ? st : launch_flatten_finish(ctx, P);
}

// grid = (slices, jobs): job blockIdx.y copied by its slices in 16-byte pieces (+ a byte tail)
__global__ void __launch_bounds__(256) device_copies_kernel(const DeviceCopyJob* __restrict__ jobs) {
  const DeviceCopyJob J = jobs[blockIdx.y];
  const size_t n16 = J.bytes / 16;
  const uint4* __restrict__ s4 = reinterpret_cast<const uint4*>(J.src);
  uint4* __restrict__ d4 = reinterpret_cast<uint4*>(J.dst);
  for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n16; i += (size_t)gridDim.x * 256) d4[i] = s4[i];
  if (blockIdx.x == 0) for (size_t i = n16 * 16 + threadIdx.x; i < J.bytes; i += 256) J.dst[i] = J.src[i];
}

int launch_device_copies(dphy_ctx* ctx, const DeviceCopyJob* d_jobs, int num_jobs, size_t max_bytes) {
  if (num_jobs <= 0) return DPHY_OK;
  const int slices = (int)std::min<size_t>(64, std::max<size_t>(1, max_bytes / (256 * 16 * 4)));
  device_copies_kernel<<<dim3(slices, num_jobs), 256, 0, ctx->stream>>>(d_jobs);
  ctx->launches += 1;
  return check_cuda(ctx, cudaGetLastError(), "device_copies_kernel");
}

int launch_flatten_lists(dphy_ctx* ctx, FlattenParams P, int first_tile, int num_tiles) {
  if (num_tiles <= 0) return DPHY_OK;
  P.tile_base = first_tile;
  flatten_events_kernel<<<num_tiles, kTile, 0, ctx->stream>>>(P);
  fold_branch_weights_kernel<<<num_tiles, kTile, 0, ctx->stream>>>(P);
  ctx->launches += 2;
  return check_cuda(ctx, cudaGetLastError(), "flatten kernels launch (lists)");
}

int launch_flatten_finish(dphy_ctx* ctx, const FlattenParams& P) {
  if (P.num_nodes == 0) return DPHY_OK;
  const int nst = (P.num_nodes + kScanTile - 1) / kScanTile, G = P.fsw_stride / 4;
  counts_scan_reduce_kernel<<<dim3(nst, G), kTile, 0, ctx->stream>>>(P);
  counts_scan_spine_kernel<<<2 * G, kTile, 0, ctx->stream>>>(P, nst);
  counts_scan_post_kernel<<<dim3(nst, G), kTile, 0, ctx->stream>>>(P);
  counts_scan_apply_kernel<<<dim3(nst, G), kTile, 0, ctx->stream>>>(P);
  flatten_ctiles_kernel<<<(P.num_ctiles + 255) / 256, 256, 0, ctx->stream>>>(P);
  ctx->launches += 5;
  return check_cuda(ctx, cudaGetLastError(), "flatten kernels launch (state counts, tile descriptors)");
}

}  // namespace dphy
