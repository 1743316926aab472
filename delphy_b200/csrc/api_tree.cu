// api_tree.cu -- the reference's wire / on-disk tree format straight to (and from) the device (SURVEY.md section 8f row 4).
//
// delphy.api.Tree (core/api.fbs:13-49) is what `.dphy` files and the WASM API carry: a FlatBuffers table with four vectors of fixed
// -size structs -- nodes, mutations sorted by branch, missation intervals sorted by branch, the reference sequence -- i.e. already
// CSR-shaped.  The reference turns it into its AoS Phylo_tree (api_tree_and_tree_info_to_phylo_tree, core/api.cpp:127-186: one
// emplace_back per mutation, one interval-set insert per interval, then fix_up_missations, core/phylo_tree.cpp:379-478, a sequential
// traversal carrying a sequence overlay and touching every missing site) and only then can anything be evaluated.  Here the host
// merely follows the table's offsets (bounds-checked: the buffer is untrusted); the struct vectors are DMA'd as they lie and
// everything else happens on the device:
//   * the struct-of-arrays split and the CSR offsets (one binary search per node over the branch column);
//   * a first flatten without from_states: the Euler-tour ranking gives every node its DFS position and subtree size;
//   * the from_states of every missation -- the one thing the format does not store.  fix_up_missations' third pass gives branch X
//     the overrides {l in X's missing intervals : state above X != ref[l]}, and the state above X at l is the `to` of the deepest
//     mutation of site l on the path root -> parent(X).  "On the path" is an interval test on DFS positions (q <= pos(P) < q + size(q)),
//     so with the mutations sorted by (site, position, list index) the mutations that can matter to an interval [s, e) are one
//     contiguous run, the ancestors among the run's entries of one site come in order of depth, and the deepest is the last that
//     passes: one warp per interval streams its run, 32 tests per step, and keeps per site the last passing entry.  The cost does
//     not depend on the depth of the tree (coalescent trees of densely sampled outbreaks are ladders thousands of levels deep) nor
//     on the number of missing sites;
//   * the reference's CHECK that every mutation starts from the state above it (core/phylo_tree.cpp:465), from the same sorted table;
//   * the forest is then re-flattened with the from_states in place (DFS order reused), by the kernels of dphy_forest_upload.
// Precondition, as for any buffer phylo_tree_to_api_tree wrote: the first two passes of fix_up_missations (bubbling common missations
// up, rewriting missations nested under an ancestor's) and its erasure of mutations on missing sites find nothing to do.  The
// cheap half is always checked (siblings share no missing site; no mutation on a site missing at its own node); the walk of every
// root path that the other half needs (O(nodes x depth)) runs with DPHY_API_TREE_CHECK_PATHS.  A buffer that fails is refused
// (DPHY_ERR_INVALID_ARGUMENT), never silently rewritten.
// The other direction (phylo_tree_to_api_tree, core/api.cpp:34-98) packs the resident host-order arrays back into the three struct
// vectors on the device; the host adds the 48-byte table header.
#include "dphy_internal.h"
#include "device_utils.cuh"

#include <algorithm>
#include <cstring>
#include <optional>
#include <vector>

namespace dphy {

namespace {

enum : uint32_t {
  kApiErrBranchRange = 1u,     // a mutation / missation interval names a branch outside [0, N)
  kApiErrNotSorted = 2u,       // records not grouped by ascending branch (core/api.fbs:44-45), or a branch's intervals not ascending and disjoint
  kApiErrNotNormal = 4u,       // fix_up_missations would rewrite the tree (see above)
  kApiErrTopology = 8u,        // parent links do not lead to the root
  kApiErrRefSeq = 16u,         // ref_seq differs from the sites table the tree is loaded against
  kApiErrFromState = 32u,      // a mutation's `from` contradicts the state above it (CHECK_EQ, core/phylo_tree.cpp:465)
};

struct ApiNode { int32_t parent, left, right; float t; };                              // core/api_generated.h:157-190
struct ApiMutation { int32_t branch, site; uint8_t from, to; int16_t pad; float t; };  // :192-236
struct ApiInterval { int32_t branch, start, end; };                                    // :238-265
static_assert(sizeof(ApiNode) == 16 && sizeof(ApiMutation) == 16 && sizeof(ApiInterval) == 12, "FlatBuffers struct sizes");

struct ApiTreeDev {
  const ApiNode* nodes; const ApiMutation* muts; const ApiInterval* ivls; const uint8_t* ref_seq;
  int32_t n, M, I, L, root;
};
struct RawOut {
  int32_t* parent; int32_t* child0; int32_t* child1; double* t;
  int32_t* mut_off; int32_t* mut_site; uint8_t* mut_from; uint8_t* mut_to; double* mut_t;
  int32_t* miss_off; int32_t* miss_start; int32_t* miss_end;
  int32_t* fs_off; int32_t* fs_site; uint8_t* fs_from;
};

// ---- struct-of-arrays split ----------------------------------------------------------------------------------------------------------------
__global__ void apitree_split_kernel(ApiTreeDev A, RawOut O, const uint8_t* __restrict__ sites_ref, uint32_t* __restrict__ status) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t err = 0;
  if (i < A.n) {
    const ApiNode nd = A.nodes[i];
    O.parent[i] = nd.parent; O.child0[i] = nd.left; O.child1[i] = nd.right; O.t[i] = (double)nd.t;    // children = {left, right} (core/api.cpp:147-151)
  }
  if (i < A.M) {
    const ApiMutation m = A.muts[i];
    if (m.branch < 0 || m.branch >= A.n) err |= kApiErrBranchRange;
    if (i > 0 && A.muts[i - 1].branch > m.branch) err |= kApiErrNotSorted;
    O.mut_site[i] = m.site; O.mut_from[i] = m.from; O.mut_to[i] = m.to; O.mut_t[i] = (double)m.t;
  }
  if (i < A.I) {
    const ApiInterval v = A.ivls[i];
    if (v.branch < 0 || v.branch >= A.n) err |= kApiErrBranchRange;
    if (i > 0) {
      const ApiInterval u = A.ivls[i - 1];
      // Interval_set::insert would merge touching intervals: a normal-form buffer has them ascending and apart
      if (u.branch > v.branch || (u.branch == v.branch && v.start <= u.end)) err |= kApiErrNotSorted;
    }
    O.miss_start[i] = v.start; O.miss_end[i] = v.end;
  }
  if (i < A.L && A.ref_seq[i] != sites_ref[i]) err |= kApiErrRefSeq;
  if (err) atomicOr(status, err);
}

// CSR offsets: off[x] = first record whose branch is >= x (the records are grouped by ascending branch)
__global__ void apitree_offsets_kernel(ApiTreeDev A, RawOut O) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x > A.n) return;
  int lo = 0, hi = A.M;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (A.muts[mid].branch < x) lo = mid + 1; else hi = mid; }
  O.mut_off[x] = lo;
  lo = 0; hi = A.I;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (A.ivls[mid].branch < x) lo = mid + 1; else hi = mid; }
  O.miss_off[x] = lo;
}

// first row of [a, b) whose interval ends after l (the intervals of a node are ascending and disjoint)
__device__ __forceinline__ int first_ending_after(const int32_t* __restrict__ e, int a, int b, int l) {
  while (a < b) { const int mid = (a + b) >> 1; if (e[mid] <= l) a = mid + 1; else b = mid; }
  return a;
}
__device__ __forceinline__ bool in_intervals(const int32_t* __restrict__ s, const int32_t* __restrict__ e, int a, int b, int l) {
  const int k = first_ending_after(e, a, b, l);
  return k < b && s[k] <= l;
}

// Always checked -- the part of "fix_up_missations finds nothing to do" that needs no path walk:
//   pass 1 (core/phylo_tree.cpp:383-398) the two children of an inner node share no missing site (else the common part moves to the parent),
//   pass 3 (:460-461) no mutation of a node lies on a site missing at that very node.
__global__ void apitree_local_form_kernel(ApiTreeDev A, RawOut O, uint32_t* __restrict__ status) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= A.n) return;
  uint32_t err = 0;
  const int c0 = O.child0[x], c1 = O.child1[x];
  if (c0 >= 0 && c0 < A.n && c1 >= 0 && c1 < A.n) {
    int a = O.miss_off[c0], b = O.miss_off[c1];
    const int ae = O.miss_off[c0 + 1], be = O.miss_off[c1 + 1];
    while (a < ae && b < be) {
      if (O.miss_start[a] < O.miss_end[b] && O.miss_start[b] < O.miss_end[a]) { err |= kApiErrNotNormal; break; }
      if (O.miss_end[a] <= O.miss_end[b]) ++a; else ++b;
    }
  }
  const int i0 = O.miss_off[x], i1 = O.miss_off[x + 1];
  if (i1 > i0)
    for (int k = O.mut_off[x]; k < O.mut_off[x + 1]; ++k) if (in_intervals(O.miss_start, O.miss_end, i0, i1, O.mut_site[k])) err |= kApiErrNotNormal;
  if (err) atomicOr(status, err);
}

// DPHY_API_TREE_CHECK_PATHS -- the part that needs every root path (runs after the first flatten, so the parent links are a tree):
//   pass 2 (:400-444) no site of a node's missations is already missing at an ancestor,
//   pass 3 (:460-461) no mutation lies on a site missing at an ancestor.
// One thread per node with a list walks to the root: O(depth) each, the reason this is opt-in.
__global__ void apitree_path_form_kernel(ApiTreeDev A, RawOut O, uint32_t* __restrict__ status) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= A.n) return;
  const int m0 = O.mut_off[x], m1 = O.mut_off[x + 1], i0 = O.miss_off[x], i1 = O.miss_off[x + 1];
  if (m1 == m0 && i1 == i0) return;
  uint32_t err = 0;
  int anc = O.parent[x], steps = 0;
  while (anc >= 0 && anc < A.n && err == 0) {
    if (++steps > A.n) { err |= kApiErrTopology; break; }
    if ((steps & 63) == 0 && *((volatile uint32_t*)status) != 0) break;      // somebody already found the buffer bad
    const int a0 = O.miss_off[anc], a1 = O.miss_off[anc + 1];
    if (a1 > a0) {
      for (int k = m0; k < m1; ++k) if (in_intervals(O.miss_start, O.miss_end, a0, a1, O.mut_site[k])) err |= kApiErrNotNormal;
      for (int k = i0; k < i1; ++k) {
        const int j = first_ending_after(O.miss_end, a0, a1, O.miss_start[k]);
        if (j < a1 && O.miss_start[j] < O.miss_end[k]) err |= kApiErrNotNormal;
      }
    }
    anc = O.parent[anc];
  }
  if (err) atomicOr(status, err);
}

// ---- the mutations sorted by (site, DFS position of their node, index in the buffer) -------------------------------------------------------
// One record per mutation: q = tree-local DFS position of its node, q_end = q + subtree size (the node is an ancestor-or-self of
// position p iff q <= p < q_end), idx = its index in the buffer (ascending inside a node == list order == time order),
// st = site << 2 | to.
struct SiteOrder {
  const int32_t* pos_of_node;      // + node_base: host id -> tree-local position (first flatten)
  const int32_t* subtree_size;     // + node_base: by position
  const int32_t* parent_pos;       // + node_base: GLOBAL position of the parent, -1 for the root
  int32_t node_base;
  int32_t* site_off;               // [L + 1] counts, then (scanned) first record of every site
  int32_t* site_fill;              // [L]
  int4* rec;                       // [M]
  int32_t* ivl_off;                // [I + 1] overrides per interval, then (scanned) where each interval's overrides go
};

__global__ void apitree_site_hist_kernel(ApiTreeDev A, SiteOrder S) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < A.M) atomicAdd(S.site_off + A.muts[i].site, 1);
}
__global__ void apitree_site_scatter_kernel(ApiTreeDev A, SiteOrder S) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A.M) return;
  const ApiMutation m = A.muts[i];
  const int q = S.pos_of_node[m.branch];
  const int slot = S.site_off[m.site] + atomicAdd(S.site_fill + m.site, 1);
  S.rec[slot] = make_int4(q, q + S.subtree_size[q], i, (m.site << 2) | (m.to & 3));
}
// the scatter lands a site's records in any order: one thread per site puts its (short) run in (q, idx) order
__global__ void apitree_site_sort_kernel(ApiTreeDev A, SiteOrder S) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= A.L) return;
  const int r0 = S.site_off[l], r1 = S.site_off[l + 1];
  for (int a = r0 + 1; a < r1; ++a) {
    const int4 v = S.rec[a];
    int b = a - 1;
    while (b >= r0) {
      const int4 u = S.rec[b];
      if (u.x < v.x || (u.x == v.x && u.z < v.z)) break;
      S.rec[b + 1] = u; --b;
    }
    S.rec[b + 1] = v;
  }
}

// CHECK_EQ(m.from, cur_seq[m.site]) (core/phylo_tree.cpp:465): every mutation starts from the state of the sequence above it -- the
// `to` of the closest mutation of the same site above it (the nearest earlier record of its site run that is an ancestor-or-self),
// else the reference sequence's.
__global__ void apitree_from_check_kernel(ApiTreeDev A, SiteOrder S, uint32_t* __restrict__ status) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= A.M) return;
  const int4 v = S.rec[j];
  const int l = v.w >> 2;
  int above = A.ref_seq[l];
  for (int b = j - 1; b >= S.site_off[l]; --b) {
    const int4 u = S.rec[b];
    if (u.x <= v.x && v.x < u.y) { above = u.w & 3; break; }
  }
  if (above != A.muts[v.z].from) atomicOr(status, kApiErrFromState);
}

// from_states (fix_up_missations pass 3, core/phylo_tree.cpp:446-459).  One warp per missation interval (X, [s, e)): the records of
// sites s .. e-1 are the run [site_off[s], site_off[e]); an entry matters iff its node is an ancestor-or-self of parent(X) (the
// root's own list included: it is applied on entering the root); of the passing entries of one site the LAST is the deepest, and it is
// an override iff its `to` differs from the reference sequence.  FILL == false counts into ivl_off[interval]; FILL == true writes the
// overrides at ivl_off[interval] + k -- in ascending site order, and a node's intervals are ascending, so every node's from_states
// come out sorted by site as the reference's flat_map keeps them.
template <bool FILL>
__global__ void __launch_bounds__(256) apitree_from_states_kernel(ApiTreeDev A, RawOut O, SiteOrder S) {
  const int iv = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (iv >= A.I) return;
  const ApiInterval v = A.ivls[iv];
  int emitted = 0;
  const int w0 = FILL ? S.ivl_off[iv] : 0;
  if (v.branch != A.root) {
    const int pp = S.parent_pos[S.pos_of_node[v.branch]] - S.node_base;       // tree-local position of parent(X)
    const int s = min(max(v.start, 0), A.L), e = min(max(v.end, s), A.L);
    const int r0 = S.site_off[s], r1 = S.site_off[e];
    int carry = -1;                                                          // st of the last passing entry seen so far (its site may continue)
    for (int base = r0; base < r1; base += 32) {
      const int j = base + lane;
      int st = -1;
      bool pass = false;
      if (j < r1) { const int4 u = S.rec[j]; st = u.w; pass = u.x <= pp && pp < u.y; }
      const uint32_t b = __ballot_sync(0xffffffffu, pass);
      if (b == 0) continue;
      // the carried entry is final once an entry of another site passes
      const int first_st = __shfl_sync(0xffffffffu, st, __ffs(b) - 1);
      if (carry >= 0 && (first_st >> 2) != (carry >> 2)) {
        if ((carry & 3) != A.ref_seq[carry >> 2]) {
          if (FILL && lane == 0) { O.fs_site[w0 + emitted] = carry >> 2; O.fs_from[w0 + emitted] = (uint8_t)(carry & 3); }
          ++emitted;
        }
      }
      // inside the chunk: a passing entry is final iff the next passing entry belongs to another site; the last one is carried on
      const uint32_t later = lane == 31 ? 0u : (b & ~((2u << lane) - 1u));
      const int next_lane = later ? __ffs(later) - 1 : lane;
      const int next_st = __shfl_sync(0xffffffffu, st, next_lane);
      const bool fin = pass && later != 0 && (next_st >> 2) != (st >> 2) && (st & 3) != A.ref_seq[st >> 2];
      const uint32_t fb = __ballot_sync(0xffffffffu, fin);
      if (FILL && fin) { const int k = w0 + emitted + __popc(fb & ((1u << lane) - 1u)); O.fs_site[k] = st >> 2; O.fs_from[k] = (uint8_t)(st & 3); }
      emitted += __popc(fb);
      carry = __shfl_sync(0xffffffffu, st, 31 - __clz(b));
    }
    if (carry >= 0 && (carry & 3) != A.ref_seq[carry >> 2]) {
      if (FILL && lane == 0) { O.fs_site[w0 + emitted] = carry >> 2; O.fs_from[w0 + emitted] = (uint8_t)(carry & 3); }
      ++emitted;
    }
  }
  if (!FILL && lane == 0) { S.ivl_off[iv] = emitted; if (iv == 0) S.ivl_off[A.I] = 0; }
}
// fs_off[x] = where the overrides of x's first interval go (a node's intervals are consecutive in the buffer)
__global__ void apitree_fs_off_kernel(ApiTreeDev A, RawOut O, SiteOrder S) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x <= A.n) O.fs_off[x] = S.ivl_off[O.miss_off[x]];
}

// ---- exclusive scan of int32 (the from-state counts -> fs_off), two levels of 1,024 x 8 tiles ------------------------------------------------
constexpr int kScanItems = 8, kScanTile = 1024 * kScanItems;
__global__ void __launch_bounds__(1024) apitree_scan_tiles_kernel(int32_t* __restrict__ v, int n, int32_t* __restrict__ tile_tot) {
  __shared__ int32_t ws[32];
  const int base = blockIdx.x * kScanTile + threadIdx.x * kScanItems;
  int32_t r[kScanItems], s = 0;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j) { r[j] = base + j < n ? v[base + j] : 0; s += r[j]; }
  int32_t total;
  const int32_t incl = block_scan_incl<int32_t, 1024>(s, ws, &total);
  int32_t run = incl - s;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j) { if (base + j < n) v[base + j] = run; run += r[j]; }
  if (threadIdx.x == 0) tile_tot[blockIdx.x] = total;
}
__global__ void __launch_bounds__(1024) apitree_scan_fix_kernel(int32_t* __restrict__ v, int n, const int32_t* __restrict__ tile_tot) {
  __shared__ int32_t carry;
  if (threadIdx.x == 0) { int32_t c = 0; for (int b = 0; b < (int)blockIdx.x; ++b) c += tile_tot[b]; carry = c; }
  __syncthreads();
  const int base = blockIdx.x * kScanTile + threadIdx.x * kScanItems;
  if (blockIdx.x > 0)
#pragma unroll
    for (int j = 0; j < kScanItems; ++j) if (base + j < n) v[base + j] += carry;
}

// ---- device -> wire format ---------------------------------------------------------------------------------------------------------------
__global__ void apitree_pack_kernel(RawTreeDev R, ApiNode* __restrict__ nodes, ApiMutation* __restrict__ muts, ApiInterval* __restrict__ ivls) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= R.num_nodes) return;
  ApiNode nd; nd.parent = R.parent[x]; nd.left = R.child0[x]; nd.right = R.child1[x]; nd.t = (float)R.t[x];   // tips: -1, -1 (core/api.cpp:64-68)
  nodes[x] = nd;
  for (int k = R.mut_off[x]; k < R.mut_off[x + 1]; ++k) {
    ApiMutation m; m.branch = x; m.site = R.mut_site[k]; m.from = R.mut_from[k]; m.to = R.mut_to[k]; m.pad = 0; m.t = (float)R.mut_t[k];
    muts[k] = m;
  }
  for (int k = R.miss_off[x]; k < R.miss_off[x + 1]; ++k) { ApiInterval v; v.branch = x; v.start = R.miss_start[k]; v.end = R.miss_end[k]; ivls[k] = v; }
}

bool pinned_host(const void* p) {
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;        // (the host parses the table header itself: device memory will not do)
}

// ---- the host side of the format: follow the table's offsets, nothing else -----------------------------------------------------------------------
uint32_t rd_u32(const uint8_t* p) { uint32_t v; std::memcpy(&v, p, 4); return v; }      // FlatBuffers is little endian, and so is every CUDA host
uint16_t rd_u16(const uint8_t* p) { uint16_t v; std::memcpy(&v, p, 2); return v; }

bool api_vector(const uint8_t* buf, int64_t len, int64_t tpos, int64_t vt, int vtsize, int slot, int64_t elem, const void** data, int64_t* count) {
  *data = nullptr; *count = 0;
  if (slot + 2 > vtsize) return true;                   // field absent == empty vector
  const int fo = rd_u16(buf + vt + slot);
  if (fo == 0) return true;
  const int64_t fpos = tpos + fo;
  if (fpos + 4 > len) return false;
  const int64_t vpos = fpos + (int64_t)rd_u32(buf + fpos);
  if (vpos + 4 > len) return false;
  const int64_t n = (int64_t)rd_u32(buf + vpos);
  if (n > INT32_MAX || vpos + 4 + n * elem > len) return false;
  *data = buf + vpos + 4; *count = n;
  return true;
}

bool parse_api_tree(const void* bufv, size_t blen, dphy_api_tree_view* out) {
  std::memset(out, 0, sizeof(*out));
  const uint8_t* buf = static_cast<const uint8_t*>(bufv);
  int64_t len = (int64_t)blen;
  if (!buf || len < 12) return false;
  const int64_t body = (int64_t)rd_u32(buf);             // FinishSizePrefixed (core/api.cpp:95)
  if (body + 4 > len) return false;
  len = body + 4;
  const int64_t tpos = 4 + (int64_t)rd_u32(buf + 4);
  if (tpos < 8 || tpos + 4 > len) return false;
  int32_t so; std::memcpy(&so, buf + tpos, 4);
  const int64_t vt = tpos - (int64_t)so;
  if (vt < 4 || vt + 4 > len) return false;
  const int vtsize = rd_u16(buf + vt), tsize = rd_u16(buf + vt + 2);
  if (vtsize < 4 || (vtsize & 1) || vt + vtsize > len || tpos + tsize > len) return false;
  for (int slot = 4; slot + 2 <= vtsize; slot += 2) { const int fo = rd_u16(buf + vt + slot); if (fo != 0 && fo + 4 > tsize) return false; }
  int64_t n = 0, L = 0;
  const void* ref = nullptr;
  if (!api_vector(buf, len, tpos, vt, vtsize, 4, 16, &out->nodes, &n)) return false;                         // VT_NODES (core/api_generated.h:269-275)
  if (!api_vector(buf, len, tpos, vt, vtsize, 6, 16, &out->mutations, &out->num_mutations)) return false;
  if (!api_vector(buf, len, tpos, vt, vtsize, 8, 12, &out->missation_intervals, &out->num_missation_intervals)) return false;
  if (!api_vector(buf, len, tpos, vt, vtsize, 10, 1, &ref, &L)) return false;
  out->ref_seq = static_cast<const uint8_t*>(ref);
  out->num_nodes = (int32_t)n; out->num_sites = (int32_t)L;
  out->root = 0;                                                                                               // the field's default (:289)
  if (12 + 2 <= vtsize && rd_u16(buf + vt + 12) != 0) std::memcpy(&out->root, buf + tpos + rd_u16(buf + vt + 12), 4);
  return true;
}

int api_status_to_error(dphy_ctx* ctx, uint32_t bits) {
  if (bits & kApiErrBranchRange) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "api tree: a mutation / missation interval names a branch outside the tree");
  if (bits & kApiErrNotSorted) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "api tree: mutations / missation intervals are not sorted by branch (intervals: ascending and apart)");
  if (bits & kApiErrRefSeq) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "api tree: ref_seq differs from the sites table's reference sequence");
  if (bits & kApiErrTopology) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "tree topology is not a binary tree rooted at `root`");
  if (bits & kApiErrNotNormal) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "api tree: not in the form phylo_tree_to_api_tree writes (fix_up_missations would rewrite its missations / mutations)");
  if (bits & kApiErrFromState) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "api tree: a mutation's `from` state contradicts the sequence above it");
  return DPHY_OK;
}

}  // namespace

int launch_scan_i32(dphy_ctx* ctx, int32_t* v, int n, int32_t* tile_tot) {
  const int nt = (n + kScanTile - 1) / kScanTile;
  apitree_scan_tiles_kernel<<<nt, 1024, 0, ctx->stream>>>(v, n, tile_tot);
  apitree_scan_fix_kernel<<<nt, 1024, 0, ctx->stream>>>(v, n, tile_tot);
  ctx->launches += 2;
  return check_cuda(ctx, cudaGetLastError(), "scan launch");
}
}  // namespace dphy

using namespace dphy;

extern "C" int dphy_api_tree_parse(const void* buf, size_t len, dphy_api_tree_view* out) {
  if (!out) return DPHY_ERR_INVALID_ARGUMENT;
  return parse_api_tree(buf, len, out) ? DPHY_OK : DPHY_ERR_INVALID_ARGUMENT;
}

extern "C" int dphy_forest_upload_api_trees(dphy_ctx* ctx, int32_t num_trees, const void* const* bufs, const size_t* lens,
                                            const int32_t* includes_run_root, const int32_t* sites_index, int32_t num_sites_tables,
                                            dphy_sites* const* sites, uint32_t flags, dphy_forest** out) {
  if (!ctx || !out || num_trees <= 0 || !bufs || !lens || !sites || num_sites_tables <= 0) return DPHY_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  cudaSetDevice(ctx->device);
  std::vector<dphy_api_tree_view> views(num_trees);
  size_t stage = 0;
  for (int k = 0; k < num_trees; ++k) {
    if (!parse_api_tree(bufs[k], lens[k], &views[k])) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "api tree: malformed FlatBuffers Tree buffer");
    const dphy_api_tree_view& v = views[k];
    if (v.num_nodes <= 0) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "empty tree");
    if (v.root < 0 || v.root >= v.num_nodes) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "root out of range");
    const int si = sites_index ? sites_index[k] : 0;
    if (si < 0 || si >= num_sites_tables || !sites[si]) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "sites_index out of range");
    if (v.num_sites != sites[si]->L) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "api tree: ref_seq differs from the sites table's reference sequence");
    stage += align_up(16 * (size_t)v.num_nodes) + align_up(16 * (size_t)v.num_mutations) + align_up(12 * (size_t)v.num_missation_intervals) + align_up((size_t)v.num_sites);
  }
  // ---- the struct vectors cross PCIe as they lie (one pinned staging pass; nothing is converted on the host) ------------------------------------
  bool staged_any = false;
  for (int k = 0; k < num_trees; ++k) staged_any = staged_any || !pinned_host(bufs[k]);
  std::optional<PinnedStage> pin;
  if (staged_any) {
    pin.emplace(ctx, stage);
    if (pin->status != DPHY_OK) return pin->status;
  }
  char* hb = pin ? pin->p : nullptr;
  std::vector<DevBlock> scratch;    // freed stream-ordered once the forest is built
  auto dalloc = [&](size_t bytes) -> char* {
    scratch.emplace_back(ctx->stream);
    return scratch.back().alloc(std::max<size_t>(bytes, 256)) ? scratch.back().p : nullptr;
  };
  char* d_in = dalloc(stage);
  uint32_t* d_status = reinterpret_cast<uint32_t*>(dalloc(256));
  if (!d_in || !d_status) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(api tree)");
  std::vector<ApiTreeDev> dev(num_trees);
  struct DirectCopy { size_t at; const void* src; size_t bytes; };
  std::vector<DirectCopy> direct_copies;
  {
    size_t o = 0;
    for (int k = 0; k < num_trees; ++k) {
      const dphy_api_tree_view& v = views[k];
      ApiTreeDev& A = dev[k];
      A.n = v.num_nodes; A.M = (int32_t)v.num_mutations; A.I = (int32_t)v.num_missation_intervals; A.L = v.num_sites; A.root = v.root;
      // a buffer in page-locked memory (dphy_host_alloc, or registered by the caller) is DMA'd from where it lies; a pageable one
      // is staged through the context's pinned slab (one pass of memcpy, the only touch the host gives the data)
      const bool direct = pinned_host(bufs[k]);
      auto put = [&](const void* src, size_t bytes) {
        const size_t at = o;
        if (bytes) {
          if (direct) direct_copies.push_back({at, src, bytes});
          else std::memcpy(hb + o, src, bytes);
        }
        o += align_up(bytes);
        return at;
      };
      A.nodes = reinterpret_cast<const ApiNode*>(d_in + put(v.nodes, 16 * (size_t)A.n));
      A.muts = reinterpret_cast<const ApiMutation*>(d_in + put(v.mutations, 16 * (size_t)A.M));
      A.ivls = reinterpret_cast<const ApiInterval*>(d_in + put(v.missation_intervals, 12 * (size_t)A.I));
      A.ref_seq = reinterpret_cast<const uint8_t*>(d_in + put(v.ref_seq, (size_t)A.L));
    }
  }
  cudaError_t ce = cudaSuccess;
  if (stage && staged_any) ce = cudaMemcpyAsync(d_in, hb, stage, cudaMemcpyHostToDevice, ctx->stream);   // (gaps left by direct buffers: garbage, overwritten next)
  pin.reset();
  for (size_t i = 0; i < direct_copies.size() && ce == cudaSuccess; ++i)
    ce = cudaMemcpyAsync(d_in + direct_copies[i].at, direct_copies[i].src, direct_copies[i].bytes, cudaMemcpyHostToDevice, ctx->stream);
  if (ce == cudaSuccess) ce = cudaMemsetAsync(d_status, 0, 256, ctx->stream);
  if (ce != cudaSuccess) return check_cuda(ctx, ce, "H2D api tree");

  // ---- per tree: struct-of-arrays split, CSR offsets, the local checks ------------------------------------------------------------------------
  std::vector<RawOut> outs(num_trees);
  std::vector<SiteOrder> ords(num_trees);
  for (int k = 0; k < num_trees; ++k) {
    const ApiTreeDev& A = dev[k];
    const size_t n = A.n, M = A.M, I = A.I, L = A.L;
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o = align_up(o + std::max<size_t>(bytes, 1)); return at; };
    const size_t a_par = take(4 * n), a_c0 = take(4 * n), a_c1 = take(4 * n), a_t = take(8 * n);
    const size_t a_moff = take(4 * (n + 1)), a_msite = take(4 * M), a_mfrom = take(M), a_mto = take(M), a_mt = take(8 * M);
    const size_t a_ioff = take(4 * (n + 1)), a_is = take(4 * I), a_ie = take(4 * I), a_foff = take(4 * (n + 1));
    const size_t a_soff = take(4 * (L + 1)), a_sfill = take(4 * L), a_rec = take(16 * M), a_ivo = take(4 * (I + 1));
    const size_t zero_from = a_foff, zero_to = a_rec;          // fs_off (an empty list per node for the first flatten), site counters
    char* nb = dalloc(o);
    if (!nb) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(api tree arrays)");
    cudaMemsetAsync(nb + zero_from, 0, zero_to - zero_from, ctx->stream);
    cudaMemsetAsync(nb + a_ivo, 0, 4 * (I + 1), ctx->stream);        // a tree without missations: F is read from ivl_off[0]
    RawOut& O = outs[k];
    O.parent = (int32_t*)(nb + a_par); O.child0 = (int32_t*)(nb + a_c0); O.child1 = (int32_t*)(nb + a_c1); O.t = (double*)(nb + a_t);
    O.mut_off = (int32_t*)(nb + a_moff); O.mut_site = (int32_t*)(nb + a_msite); O.mut_from = (uint8_t*)(nb + a_mfrom);
    O.mut_to = (uint8_t*)(nb + a_mto); O.mut_t = (double*)(nb + a_mt);
    O.miss_off = (int32_t*)(nb + a_ioff); O.miss_start = (int32_t*)(nb + a_is); O.miss_end = (int32_t*)(nb + a_ie);
    O.fs_off = (int32_t*)(nb + a_foff); O.fs_site = nullptr; O.fs_from = nullptr;
    SiteOrder& S = ords[k];
    S.site_off = (int32_t*)(nb + a_soff); S.site_fill = (int32_t*)(nb + a_sfill); S.rec = (int4*)(nb + a_rec); S.ivl_off = (int32_t*)(nb + a_ivo);
    const int si = sites_index ? sites_index[k] : 0;
    const int most = std::max({A.n, A.M, A.I, A.L});
    apitree_split_kernel<<<(most + 255) / 256, 256, 0, ctx->stream>>>(A, O, sites[si]->d_ref, d_status);
    apitree_offsets_kernel<<<(A.n + 1 + 255) / 256, 256, 0, ctx->stream>>>(A, O);
    apitree_local_form_kernel<<<(A.n + 127) / 128, 128, 0, ctx->stream>>>(A, O, d_status);
    ctx->launches += 3;
  }
  int st = check_cuda(ctx, cudaGetLastError(), "api tree kernels");
  uint32_t h_status = 0;
  auto read_status = [&]() {
    int s2 = check_cuda(ctx, cudaMemcpyAsync(&h_status, d_status, 4, cudaMemcpyDeviceToHost, ctx->stream), "D2H");
    if (s2 == DPHY_OK) s2 = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "api tree");
    return s2 != DPHY_OK ? s2 : api_status_to_error(ctx, h_status);
  };
  // the length of the root's mutation list (the flatten wants it on the host); the status word
  std::vector<int32_t> h_root(2 * (size_t)num_trees, 0);
  for (int k = 0; k < num_trees && st == DPHY_OK; ++k)
    st = check_cuda(ctx, cudaMemcpyAsync(&h_root[2 * k], outs[k].mut_off + dev[k].root, 8, cudaMemcpyDeviceToHost, ctx->stream), "D2H");
  if (st == DPHY_OK) st = read_status();
  if (st != DPHY_OK) return st;

  // ---- first flatten, without from_states: topology / range validation of an upload, DFS positions and subtree sizes -------------------------------
  std::vector<dphy_emat_host> ev(num_trees);
  std::vector<TreeTotals> totals(num_trees);
  for (int k = 0; k < num_trees; ++k) {
    const ApiTreeDev& A = dev[k];
    const RawOut& O = outs[k];
    dphy_emat_host& e = ev[k];
    std::memset(&e, 0, sizeof(e));
    e.num_nodes = A.n; e.root = A.root; e.includes_run_root = includes_run_root ? includes_run_root[k] : 1;
    e.parent = O.parent; e.child0 = O.child0; e.child1 = O.child1; e.t = O.t;
    e.mut_off = O.mut_off; e.mut_site = O.mut_site; e.mut_from = O.mut_from; e.mut_to = O.mut_to; e.mut_t = O.mut_t;
    e.miss_off = O.miss_off; e.miss_start = O.miss_start; e.miss_end = O.miss_end;
    e.fs_off = O.fs_off; e.fs_site = nullptr; e.fs_from = nullptr;
    totals[k] = {A.M, A.I, 0, (int64_t)h_root[2 * k + 1] - (int64_t)h_root[2 * k]};
  }
  dphy_forest* fo = nullptr;
  st = forest_from_device_arrays(ctx, num_trees, ev.data(), totals.data(), sites_index, num_sites_tables, sites, &fo);
  if (st != DPHY_OK) return st;

  // ---- from_states (and the `from` CHECK) off the site-sorted mutation table ---------------------------------------------------------------------
  bool any_fs = false;
  for (int k = 0; k < num_trees; ++k) {
    const ApiTreeDev& A = dev[k];
    RawOut& O = outs[k];
    SiteOrder& S = ords[k];
    S.node_base = fo->trees[k].node_base;
    S.pos_of_node = fo->h.pos_of_node + S.node_base; S.subtree_size = fo->h.subtree_size + S.node_base; S.parent_pos = fo->h.parent_pos + S.node_base;
    if (flags & DPHY_API_TREE_CHECK_PATHS) { apitree_path_form_kernel<<<(A.n + 127) / 128, 128, 0, ctx->stream>>>(A, O, d_status); ++ctx->launches; }
    int32_t* tile_tot = reinterpret_cast<int32_t*>(dalloc(4 * (size_t)(std::max(A.L, A.I) + 1 + kScanTile) / kScanTile * 2 + 256));
    if (!tile_tot) { st = set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(api tree scan)"); break; }
    if (A.M > 0) {
      apitree_site_hist_kernel<<<(A.M + 255) / 256, 256, 0, ctx->stream>>>(A, S);
      const int nt = (A.L + 1 + kScanTile - 1) / kScanTile;
      apitree_scan_tiles_kernel<<<nt, 1024, 0, ctx->stream>>>(S.site_off, A.L + 1, tile_tot);
      apitree_scan_fix_kernel<<<nt, 1024, 0, ctx->stream>>>(S.site_off, A.L + 1, tile_tot);
      apitree_site_scatter_kernel<<<(A.M + 255) / 256, 256, 0, ctx->stream>>>(A, S);
      apitree_site_sort_kernel<<<(A.L + 127) / 128, 128, 0, ctx->stream>>>(A, S);
      apitree_from_check_kernel<<<(A.M + 127) / 128, 128, 0, ctx->stream>>>(A, S, d_status);
      ctx->launches += 6;
    }
    if (A.I > 0) {
      apitree_from_states_kernel<false><<<(int)(((int64_t)A.I * 32 + 255) / 256), 256, 0, ctx->stream>>>(A, O, S);
      const int nt = (A.I + 1 + kScanTile - 1) / kScanTile;
      apitree_scan_tiles_kernel<<<nt, 1024, 0, ctx->stream>>>(S.ivl_off, A.I + 1, tile_tot);
      apitree_scan_fix_kernel<<<nt, 1024, 0, ctx->stream>>>(S.ivl_off, A.I + 1, tile_tot);
      ctx->launches += 3;
    }
  }
  if (st == DPHY_OK) st = check_cuda(ctx, cudaGetLastError(), "api tree from_states (count)");
  std::vector<int32_t> h_F(num_trees, 0);
  for (int k = 0; k < num_trees && st == DPHY_OK; ++k)
    st = check_cuda(ctx, cudaMemcpyAsync(&h_F[k], ords[k].ivl_off + dev[k].I, 4, cudaMemcpyDeviceToHost, ctx->stream), "D2H");   // I == 0: the zeroed word
  if (st == DPHY_OK) st = read_status();
  for (int k = 0; k < num_trees && st == DPHY_OK; ++k) {
    const ApiTreeDev& A = dev[k];
    RawOut& O = outs[k];
    const size_t F = (size_t)h_F[k];
    if (F == 0) continue;
    any_fs = true;
    char* fb = dalloc(align_up(4 * F) + align_up(F));
    if (!fb) { st = set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(api tree from_states)"); break; }
    O.fs_site = (int32_t*)fb; O.fs_from = (uint8_t*)(fb + align_up(4 * F));
    apitree_from_states_kernel<true><<<(int)(((int64_t)A.I * 32 + 255) / 256), 256, 0, ctx->stream>>>(A, O, ords[k]);
    apitree_fs_off_kernel<<<(A.n + 1 + 255) / 256, 256, 0, ctx->stream>>>(A, O, ords[k]);
    ctx->launches += 2;
    ev[k].fs_site = O.fs_site; ev[k].fs_from = O.fs_from;
    totals[k].fs = (int64_t)F;
  }
  if (st == DPHY_OK) st = check_cuda(ctx, cudaGetLastError(), "api tree from_states (fill)");
  // ---- second flatten with the from_states in place; the links did not change, so the DFS order is reused (no Euler-tour ranking) ----------------
  if (st == DPHY_OK && any_fs) st = rebuild_forest_from_device(ctx, fo, ev.data(), totals.data(), true);
  scratch.clear();
  if (st != DPHY_OK) { dphy_forest_destroy(ctx, fo); return st; }
  *out = fo;
  return DPHY_OK;
}

extern "C" int dphy_forest_tree_counts(dphy_ctx* ctx, dphy_forest* fo, int32_t tree, dphy_tree_counts* out) {
  if (!ctx || !fo || !out) return DPHY_ERR_INVALID_ARGUMENT;
  if (tree < 0 || tree >= fo->h.num_trees || (int)fo->raw.size() != fo->h.num_trees) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "tree index out of range");
  const RawTreeDev& R = fo->raw[tree];
  out->num_nodes = R.num_nodes; out->root = R.root; out->num_mutations = R.num_muts; out->num_missation_intervals = R.num_ivls; out->num_from_states = R.num_fs;
  return DPHY_OK;
}

extern "C" int dphy_forest_download_tree(dphy_ctx* ctx, dphy_forest* fo, int32_t tree, dphy_emat_host* out) {
  if (!ctx || !fo || !out) return DPHY_ERR_INVALID_ARGUMENT;
  if (tree < 0 || tree >= fo->h.num_trees || (int)fo->raw.size() != fo->h.num_trees) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "tree index out of range");
  cudaSetDevice(ctx->device);
  const RawTreeDev& R = fo->raw[tree];
  const size_t n = R.num_nodes, M = R.num_muts, I = R.num_ivls, F = R.num_fs;
  out->num_nodes = R.num_nodes; out->root = R.root; out->includes_run_root = fo->trees[tree].includes_run_root; out->reserved = 0;
  struct J { const void* dst; const void* src; size_t bytes; };
  const J jobs[] = {
    {out->parent, R.parent, 4 * n}, {out->child0, R.child0, 4 * n}, {out->child1, R.child1, 4 * n}, {out->t, R.t, 8 * n},
    {out->mut_off, R.mut_off, 4 * (n + 1)}, {out->mut_site, R.mut_site, 4 * M}, {out->mut_from, R.mut_from, M}, {out->mut_to, R.mut_to, M}, {out->mut_t, R.mut_t, 8 * M},
    {out->miss_off, R.miss_off, 4 * (n + 1)}, {out->miss_start, R.miss_start, 4 * I}, {out->miss_end, R.miss_end, 4 * I},
    {out->fs_off, R.fs_off, 4 * (n + 1)}, {out->fs_site, R.fs_site, 4 * F}, {out->fs_from, R.fs_from, F}};
  for (const J& j : jobs) {
    if (j.bytes == 0) continue;
    if (!j.dst) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "download_tree: a NULL output array");
    DPHY_CUDA(ctx, cudaMemcpyAsync(const_cast<void*>(j.dst), j.src, j.bytes, cudaMemcpyDeviceToHost, ctx->stream));
  }
  DPHY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return DPHY_OK;
}

extern "C" int64_t dphy_forest_write_api_tree(dphy_ctx* ctx, dphy_forest* fo, int32_t tree, void* outv, size_t cap) {
  if (!ctx || !fo) return DPHY_ERR_INVALID_ARGUMENT;
  if (tree < 0 || tree >= fo->h.num_trees || (int)fo->raw.size() != fo->h.num_trees) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "tree index out of range");
  cudaSetDevice(ctx->device);
  const RawTreeDev& R = fo->raw[tree];
  const dphy_sites* s = fo->sites[fo->sites_index[tree]];
  const int64_t n = R.num_nodes, M = R.num_muts, I = R.num_ivls, L = s->L;
  // [size u32][root uoffset][vtable: 14, 24, 4, 8, 12, 16, 20 + 2 B padding][table: soffset, 4 vector uoffsets, root_node][the four vectors]
  const int64_t vt = 8, tpos = 24, v_nodes = 48, v_muts = v_nodes + 4 + 16 * n, v_ivls = v_muts + 4 + 16 * M, v_ref = v_ivls + 4 + 12 * I,
                total = (v_ref + 4 + L + 3) / 4 * 4;
  if (!outv) return total;                                // size query
  if ((int64_t)cap < total) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "write_api_tree: buffer too small");
  DevBlock blk(ctx->stream);
  if (!blk.alloc((size_t)total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(api tree out)");
  char* d = blk.p;
  cudaMemsetAsync(d, 0, (size_t)total, ctx->stream);
  apitree_pack_kernel<<<(int)((n + 127) / 128), 128, 0, ctx->stream>>>(R, reinterpret_cast<ApiNode*>(d + v_nodes + 4), reinterpret_cast<ApiMutation*>(d + v_muts + 4),
                                                                    reinterpret_cast<ApiInterval*>(d + v_ivls + 4));
  ++ctx->launches;
  cudaError_t ce = cudaGetLastError();
  if (ce == cudaSuccess && L > 0) ce = cudaMemcpyAsync(d + v_ref + 4, s->d_ref, (size_t)L, cudaMemcpyDeviceToDevice, ctx->stream);
  if (ce != cudaSuccess) return check_cuda(ctx, ce, "write_api_tree");
  // through the context's pinned slab: a device-to-pageable copy is staged by the driver in small pieces (measured 4x slower)
  PinnedStage pin(ctx, (size_t)total);
  if (pin.status != DPHY_OK) return DPHY_ERR_OUT_OF_MEMORY;
  ce = cudaMemcpyAsync(pin.p, d, (size_t)total, cudaMemcpyDeviceToHost, ctx->stream);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
  blk.reset();
  if (ce != cudaSuccess) return check_cuda(ctx, ce, "write_api_tree");
  std::memcpy(outv, pin.p, (size_t)total);
  uint8_t* o = static_cast<uint8_t*>(outv);
  auto w32 = [&](int64_t at, uint32_t v) { std::memcpy(o + at, &v, 4); };
  auto w16 = [&](int64_t at, uint16_t v) { std::memcpy(o + at, &v, 2); };
  w32(0, (uint32_t)(total - 4)); w32(4, (uint32_t)(tpos - 4));
  w16(vt, 14); w16(vt + 2, 24);
  for (int i = 0; i < 5; ++i) w16(vt + 4 + 2 * i, (uint16_t)(4 + 4 * i));
  w32(tpos, (uint32_t)(tpos - vt));
  w32(tpos + 4, (uint32_t)(v_nodes - (tpos + 4))); w32(tpos + 8, (uint32_t)(v_muts - (tpos + 8)));
  w32(tpos + 12, (uint32_t)(v_ivls - (tpos + 12))); w32(tpos + 16, (uint32_t)(v_ref - (tpos + 16)));
  w32(tpos + 20, (uint32_t)R.root);
  w32(v_nodes, (uint32_t)n); w32(v_muts, (uint32_t)M); w32(v_ivls, (uint32_t)I); w32(v_ref, (uint32_t)L);
  return total;
}
