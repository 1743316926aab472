// kernels_place.cu -- batched maximum-parsimony placement of new samples on a device-resident tree (sm_100a).
//
// The question build_usher_like_tree asks per tip (core/phylo_tree.cpp:918-932) and UShER-style placement asks per new sequence:
// over the regions of an unbounded study of the sample from the root (Spr_study_builder::seed_fill_from with X == k_no_node,
// t_X == DBL_MAX, core/spr_study.cpp:9-128), the least min_muts, how many regions attain it and which is first in emission order --
// without materialising the ~N + M regions of the study or an O(L) table of the sample.
//
// Regions are numbered in emission order: the root region (root, n_root) is 0, then every non-root node v in device order (the
// builder's LIFO order, children[1] first) contributes (v, 0..n_v) at base(v) = (v - root) + mut_off[v] - mut_off[root + 1].  The
// regions below v are the block [base(v), end(v)), end(v) = base(v + subtree_size(v)), and the k-th mutation of v lies above
// [base(v) + k + 1, end(v)); the root's own list lies above every region.  With the Hamming-potential restatement (SURVEY.md
// section 8a, a12), for a sample with deltas D from the reference and missing set Mx:
//   min_muts(r) = B + Hr[r] + sum over m in A above r of c(m)
//   Hr[r] = sum of dref(m) over the mutations above r,    dref(m) = [to != ref_l] - [from != ref_l]
//   B = #{l in D \ Mx : x_l != ref_l},  A = mutations at sites in D u Mx,  c(m) = dx(m) - dref(m), dx(m) = 0 on Mx
// (true when every mutation's `from` is the state above it, which the builder's delta arithmetic assumes as well).
// Hr is study-independent: it lives in a min / count segment tree next to a site-sorted table of the mutations' region ranges (the
// per-tree index, built once per forest).  A sample's correction is piecewise constant between the 2|A| range endpoints: sort them,
// sweep, and ask the segment tree for (min, count) per piece -- O(|A| log R) per sample instead of O(R + L).
//
// Dated placement (remove_regions_in_Xs_future with a per-sample t_X, core/spr_study.cpp:211-224) keeps the regions with
// t_min < t_X: the first K = #{t_min < t_X} regions in (t_min, region) order.  A sample with K == R runs the path above unchanged;
// one with K < R asks the same per-piece questions restricted to the kept regions, of the dated part of the index: a merge-sort tree
// over region index whose nodes list their regions in t_min order, with prefix (min, count) of Hr and fractional-cascading left
// counts, so that a range query or a restricted find-first is still O(log R).
#include "dphy_internal.h"
#include "device_utils.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <algorithm>
#include <cfloat>
#include <climits>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

namespace dphy {

// ---- per-tree index --------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int region_base(const ForestDev& f, int nb, int p) { return (p - nb) + f.mut_off[p] - f.mut_off[nb + 1]; }

__global__ void place_site_hist_kernel(ForestDev f, int m0, int M, int32_t* __restrict__ site_off) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < M) atomicAdd(site_off + f.mut_site[m0 + i], 1);
}

// one thread per mutation: its node (binary search on the CSR offsets), its region range, its reference potential; scattered into
// its site's run of the table and added to the difference array of Hr
__global__ void place_site_scatter_kernel(ForestDev f, int nb, int N, int R, int m0, int M, const uint8_t* __restrict__ ref,
                                          const int32_t* __restrict__ site_off, int32_t* __restrict__ fill, int4* __restrict__ rec,
                                          int32_t* __restrict__ diff) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  const int g = m0 + i;
  int lo = nb, hi = nb + N - 1;                     // last node whose list starts at or before g
  while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (f.mut_off[mid] <= g) lo = mid; else hi = mid - 1; }
  const int p = lo;
  int a = 0, b = R;
  if (p != nb) { a = region_base(f, nb, p) + (g - f.mut_off[p]) + 1; b = region_base(f, nb, p + f.subtree_size[p]); }
  const int site = f.mut_site[g], code = f.mut_code[g], from = (code >> 2) & 3, to = code & 3, rl = ref[site];
  const int dref = (int)(to != rl) - (int)(from != rl);
  const int slot = site_off[site] + atomicAdd(fill + site, 1);
  rec[slot] = make_int4(a, b, (from << 2) | to, dref);
  if (dref) { atomicAdd(diff + a, dref); atomicAdd(diff + b, -dref); }
}

__device__ __forceinline__ int2 seg_comb(int2 a, int2 b) {
  const int m = min(a.x, b.x);
  return make_int2(m, (a.x == m ? a.y : 0) + (b.x == m ? b.y : 0));
}
// leaves: Hr[r] = inclusive prefix of the difference array = the exclusive scan at r + 1; padding leaves never win
__global__ void place_seg_leaves_kernel(const int32_t* __restrict__ scanned, int R, int P2, int2* __restrict__ seg) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < P2) seg[P2 + r] = r < R ? make_int2(scanned[r + 1], 1) : make_int2(INT_MAX, 0);
}
__global__ void place_seg_level_kernel(int2* __restrict__ seg, int lo) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < lo) { const int v = lo + i; seg[v] = seg_comb(seg[2 * v], seg[2 * v + 1]); }
}

// ---- segment tree queries ----------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int2 seg_query(const int2* __restrict__ seg, int P2, int l, int r) {
  int2 acc = make_int2(INT_MAX, 0);
  for (l += P2, r += P2; l < r; l >>= 1, r >>= 1) {
    if (l & 1) acc = seg_comb(acc, __ldg(seg + l++));
    if (r & 1) acc = seg_comb(acc, __ldg(seg + --r));
  }
  return acc;
}
// first leaf at or after l whose Hr is <= target (the caller knows one exists before its segment ends): climb to the next subtree to
// the right until one holds such a leaf, then descend to its leftmost
__device__ __forceinline__ int seg_find_first(const int2* __restrict__ seg, int P2, int l, int target) {
  int v = P2 + l;
  while (__ldg(seg + v).x > target) {
    while (v & 1) v >>= 1;
    if (v == 0) return -1;
    ++v;
  }
  while (v < P2) v = __ldg(seg + 2 * v).x <= target ? 2 * v : 2 * v + 1;
  return v - P2;
}

// ---- dated part: merge-sort tree over region index, entries of every node in t_min order -----------------------------------------------
// The node of level s at [a, a + 2^s) keeps its entries at [a, a + 2^s) of the level's tables.  With K = #{regions: t_min < t_X} the
// kept regions are the first K in t_min order, so the kept entries of every node are a prefix of its list; its length k is carried
// from the root (k = K) to the children through lc in O(1) per level.
struct DatedView { const int2* seg; const int32_t* lc; const int2* pre; int32_t P2; };

// (min Hr, count) over the first k entries of node (s, a)
__device__ __forceinline__ int2 dated_node(const DatedView& D, int s, int a, int k) {
  if (k <= 0) return make_int2(INT_MAX, 0);
  if (s == 0) return __ldg(D.seg + D.P2 + a);
  return __ldg(D.pre + (size_t)(s - 1) * D.P2 + a + k - 1);
}
// how many of the first k entries of node (s >= 1, a) come from its left child
__device__ __forceinline__ int dated_left(const DatedView& D, int s, int a, int k) {
  return k > 0 ? __ldg(D.lc + (size_t)(s - 1) * D.P2 + a + k - 1) : 0;
}

// (min, count) of Hr over the kept regions of [l, r), l < r: descend to the node where [l, r) splits, then walk its two boundary paths
__device__ int2 dated_query(const DatedView& D, int lg, int K, int l, int r) {
  int s = lg, a = 0, k = K;
  for (;;) {
    if (k == 0) return make_int2(INT_MAX, 0);
    if (l == a && r == a + (1 << s)) return dated_node(D, s, a, k);
    const int h = 1 << (s - 1), kl = dated_left(D, s, a, k);
    if (r <= a + h) { --s; k = kl; }
    else if (l >= a + h) { --s; a += h; k -= kl; }
    else break;
  }
  const int h = 1 << (s - 1), kl = dated_left(D, s, a, k);
  int2 acc = make_int2(INT_MAX, 0);
  for (int ss = s - 1, aa = a, kk = kl; kk > 0;) {              // [l, aa + 2^ss) in node (ss, aa)
    if (l == aa) { acc = seg_comb(acc, dated_node(D, ss, aa, kk)); break; }
    const int hh = 1 << (ss - 1), kkl = dated_left(D, ss, aa, kk);
    if (l < aa + hh) { acc = seg_comb(acc, dated_node(D, ss - 1, aa + hh, kk - kkl)); kk = kkl; }
    else { aa += hh; kk -= kkl; }
    --ss;
  }
  for (int ss = s - 1, aa = a + h, kk = k - kl; kk > 0;) {      // [aa, r) in node (ss, aa)
    if (r == aa + (1 << ss)) { acc = seg_comb(acc, dated_node(D, ss, aa, kk)); break; }
    const int hh = 1 << (ss - 1), kkl = dated_left(D, ss, aa, kk);
    if (r > aa + hh) { acc = seg_comb(acc, dated_node(D, ss - 1, aa, kkl)); aa += hh; kk -= kkl; }
    else kk = kkl;
    --ss;
  }
  return acc;
}

// first kept region at or after l whose Hr is <= target (seg_find_first restricted to the kept regions): on the path from the root
// to leaf l, the deepest right sibling holding such a region is the nearest; descend from it to its leftmost one
__device__ int dated_find_first(const DatedView& D, int lg, int K, int l, int target) {
  int s = lg, a = 0, k = K, cs = -1, ca = 0, ck = 0;
  while (s > 0 && k > 0) {
    const int h = 1 << (s - 1), kl = dated_left(D, s, a, k);
    if (l < a + h) {
      if (k > kl && dated_node(D, s - 1, a + h, k - kl).x <= target) { cs = s - 1; ca = a + h; ck = k - kl; }
      k = kl;
    } else { a += h; k -= kl; }
    --s;
  }
  if (s == 0 && k > 0 && __ldg(D.seg + D.P2 + a).x <= target) return a;
  if (cs < 0) return -1;
  for (s = cs, a = ca, k = ck; s > 0; --s) {
    const int kl = dated_left(D, s, a, k);
    if (dated_node(D, s - 1, a, kl).x <= target) k = kl;
    else { a += 1 << (s - 1); k -= kl; }
  }
  return a;
}

// ---- dated part: build ------------------------------------------------------------------------------------------------------------------
// the key of every region (remove_regions_in_Xs_future compares it with t_X): -DBL_MAX for the root region, t[parent] for (v, 0),
// mut_t[j - 1] for (v, j); one thread per node
__global__ void place_tkey_kernel(ForestDev f, int nb, int N, double* __restrict__ key, int32_t* __restrict__ idx) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  if (i == 0) { key[0] = -DBL_MAX; idx[0] = 0; return; }
  const int p = nb + i, b = region_base(f, nb, p), m0 = f.mut_off[p], n = f.mut_off[p + 1] - m0;
  key[b] = f.t[f.parent_pos[p]]; idx[b] = b;
  for (int j = 1; j <= n; ++j) { key[b + j] = f.mut_t[m0 + j - 1]; idx[b + j] = b + j; }
}

// doubles as monotone unsigned integers (atomicMax of the largest key)
__device__ __forceinline__ unsigned long long ordered_bits(double x) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(x);
  return (u >> 63) ? ~u : u | (1ull << 63);
}
__global__ void place_tkey_max_kernel(ForestDev f, int nb, int N, unsigned long long* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long m = ordered_bits(-DBL_MAX);
  if (i > 0 && i < N) {
    const int p = nb + i;
    m = max(m, ordered_bits(f.t[f.parent_pos[p]]));
    for (int j = f.mut_off[p]; j < f.mut_off[p + 1]; ++j) m = max(m, ordered_bits(f.mut_t[j]));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

__global__ void place_pad_list_kernel(int32_t* __restrict__ list, int R, int P2) {
  const int i = R + blockIdx.x * blockDim.x + threadIdx.x;
  if (i < P2) list[i] = i;                 // padding regions rank after every region and are never kept
}

struct DatedAcc { int lc, m, c; };
struct DatedComb {
  __device__ __forceinline__ DatedAcc operator()(const DatedAcc& a, const DatedAcc& b) const {
    const int m = min(a.m, b.m);
    return DatedAcc{a.lc + b.lc, m, (a.m == m ? a.c : 0) + (b.m == m ? b.c : 0)};
  }
};
struct SameNode {                          // scan keys are list positions; a node of level s is an aligned run of 2^s of them
  int s;
  __device__ __forceinline__ bool operator()(int a, int b) const { return (a >> s) == (b >> s); }
};
// level s: entry i of the level's list -> (comes from the left child, Hr, 1); padding leaves are (INT_MAX, 0) and never win
__global__ void place_dated_vals_kernel(const int32_t* __restrict__ list, const int2* __restrict__ seg, int P2, int s,
                                        DatedAcc* __restrict__ vals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P2) return;
  const int r = list[i];
  const int2 q = seg[P2 + r];
  vals[i] = DatedAcc{((r >> (s - 1)) & 1) ^ 1, q.x, q.y};
}
// the scanned level: its two tables, and its list stably partitioned into the lists of its children (the next level's list)
__global__ void place_dated_level_kernel(const int32_t* __restrict__ list, const DatedAcc* __restrict__ acc, int P2, int s,
                                         int32_t* __restrict__ lc, int2* __restrict__ pre, int32_t* __restrict__ next) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P2) return;
  const DatedAcc v = acc[i];
  lc[i] = v.lc;
  pre[i] = make_int2(v.m, v.c);
  const int r = list[i], a = i & ~((1 << s) - 1), h = 1 << (s - 1);
  next[((r >> (s - 1)) & 1) ? a + h + (i - a) - v.lc : a + v.lc - 1] = r;
}

// ---- stable warp-level LSD radix sort of (key, value) pairs in global scratch -----------------------------------------------------------
// Sorts n pairs by key bits [0, bits), ping-ponging between (k0, v0) and (k1, v1); returns true if the result is in (k1, v1).  Equal
// keys keep their order (a chunk of 32 is scattered in lane order: rank among the lanes of the same digit).
__device__ bool warp_radix_sort(uint32_t* k0, uint32_t* v0, uint32_t* k1, uint32_t* v1, int n, int bits, int* cnt, int lane) {
  bool alt = false;
  if (n < 2) return alt;
  for (int sh = 0; sh < bits; sh += 8) {
    const uint32_t* ks = alt ? k1 : k0; const uint32_t* vs = alt ? v1 : v0;
    uint32_t* kd = alt ? k0 : k1; uint32_t* vd = alt ? v0 : v1;
    for (int d = lane; d < 256; d += 32) cnt[d] = 0;
    __syncwarp();
    for (int i = lane; i < n; i += 32) atomicAdd(cnt + ((ks[i] >> sh) & 255), 1);
    __syncwarp();
    int loc[8], s = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) { loc[j] = cnt[lane * 8 + j]; s += loc[j]; }
    int run = warp_scan_incl(s, lane) - s;
#pragma unroll
    for (int j = 0; j < 8; ++j) { cnt[lane * 8 + j] = run; run += loc[j]; }
    __syncwarp();
    for (int i0 = 0; i0 < n; i0 += 32) {
      const int i = i0 + lane;
      const bool act = i < n;
      const uint32_t key = act ? ks[i] : 0u, val = act ? vs[i] : 0u;
      const int d = act ? (int)((key >> sh) & 255) : 256 + lane;
      const unsigned peers = __match_any_sync(0xffffffffu, d);
      const int rank = __popc(peers & ((1u << lane) - 1u));
      const int base = act ? cnt[d] : 0;
      __syncwarp();
      if (act && rank == 0) cnt[d] = base + __popc(peers);
      __syncwarp();
      if (act) { kd[base + rank] = key; vd[base + rank] = val; }
    }
    __syncwarp();
    alt = !alt;
  }
  return alt;
}

__device__ __forceinline__ int warp_min(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

struct PlaceParams {
  ForestDev f;
  int32_t nb, N, R, P2, L, site_bits, pos_bits, can_change_root, max_best, s0, s1, lg;
  const int32_t* site_off; const int4* rec; const int2* seg; const uint8_t* ref;
  const double* t_X;             // [S] date limits (null: undated call)
  const double* tkey;            // the dated part (null: not needed by this call, every K == R) ...
  const int32_t* lc; const int2* pre;
  const int32_t* delta_off; const int32_t* delta_site; const uint8_t* delta_to;
  const int32_t* miss_off; const int32_t* miss_start; const int32_t* miss_end;
  const int64_t* scr_off;        // [S + 1] words of scratch per sample (prefix); a batch uses scratch + scr_off[k] - scr_off[s0]
  uint32_t* scratch;
  dphy_placement* out;
  dphy_candidate_region* best;
};

// region index -> (device position, mut_idx) and the record the study would emit for it
__device__ __forceinline__ dphy_candidate_region place_region_record(const PlaceParams& P, int r, double tX) {
  const ForestDev& f = P.f;
  dphy_candidate_region c;
  if (r == 0) {
    c.branch = f.node_id[P.nb]; c.mut_idx = f.mut_off[P.nb + 1] - f.mut_off[P.nb]; c.t_min = -DBL_MAX; c.t_max = f.t[P.nb];
  } else {
    int lo = P.nb + 1, hi = P.nb + P.N - 1;
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (region_base(f, P.nb, mid) <= r) lo = mid; else hi = mid - 1; }
    const int j = r - region_base(f, P.nb, lo), m0 = f.mut_off[lo], n = f.mut_off[lo + 1] - m0;
    c.branch = f.node_id[lo]; c.mut_idx = j;
    c.t_min = j == 0 ? f.t[f.parent_pos[lo]] : f.mut_t[m0 + j - 1];
    c.t_max = j == n ? f.t[lo] : f.mut_t[m0 + j];
  }
  if (P.t_X && c.t_max > tX) c.t_max = tX;
  c.min_muts = 0; c.pad_ = 0; c.log_W_over_Wmax = 0.0; c.W_over_Wmax = 0.0;
  return c;
}

// K == R (nothing dropped): the undated segment tree
__device__ __forceinline__ int2 place_query(const PlaceParams& P, int K, int l, int r) {
  return K == P.R ? seg_query(P.seg, P.P2, l, r) : dated_query(DatedView{P.seg, P.lc, P.pre, P.P2}, P.lg, K, l, r);
}
__device__ __forceinline__ int place_find_first(const PlaceParams& P, int K, int l, int target) {
  return K == P.R ? seg_find_first(P.seg, P.P2, l, target) : dated_find_first(DatedView{P.seg, P.lc, P.pre, P.P2}, P.lg, K, l, target);
}

constexpr int kPlaceWarps = 8;

// one warp per sample
__global__ void __launch_bounds__(kPlaceWarps * 32, 2) place_samples_kernel(PlaceParams P) {
  __shared__ int s_cnt[kPlaceWarps][256];
  __shared__ int s_n[kPlaceWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int k = P.s0 + blockIdx.x * kPlaceWarps + warp;
  if (k >= P.s1) return;
  int* cnt = s_cnt[warp];
  const int d0 = P.delta_off[k], nd = P.delta_off[k + 1] - d0;
  const int i0 = P.miss_off[k], ni = P.miss_off[k + 1] - i0;
  const int64_t words = P.scr_off[k + 1] - P.scr_off[k];
  const int E = (int)(words / 4 - nd - ni);
  uint32_t* ek0 = P.scratch + (P.scr_off[k] - P.scr_off[P.s0]);
  uint32_t *ev0 = ek0 + E, *ek1 = ev0 + E, *ev1 = ek1 + E;
  uint32_t *dk0 = ev1 + E, *dv0 = dk0 + nd, *dk1 = dv0 + nd, *dv1 = dk1 + nd;
  uint32_t *ik0 = dv1 + nd, *iv0 = ik0 + ni, *ik1 = iv0 + ni, *iv1 = ik1 + ni;

  // (1) missing intervals sorted by start, then cut to disjoint pieces: piece i = [max(start_i, max end before i), end_i)
  // (empty pieces keep start == end; starts stay ascending, so a site's piece is found by one binary search)
  for (int i = lane; i < ni; i += 32) { ik0[i] = (uint32_t)P.miss_start[i0 + i]; iv0[i] = (uint32_t)P.miss_end[i0 + i]; }
  __syncwarp();
  const bool ialt = warp_radix_sort(ik0, iv0, ik1, iv1, ni, P.site_bits, cnt, lane);
  uint32_t* is = ialt ? ik1 : ik0;
  uint32_t* ie = ialt ? iv1 : iv0;
  int carry = 0;
  for (int b0 = 0; b0 < ni; b0 += 32) {
    const int i = b0 + lane;
    const int s = i < ni ? (int)is[i] : 0, e = i < ni ? (int)ie[i] : 0;
    int incl = e;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl = max(incl, u); }
    int excl = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) excl = 0;
    const int s2 = max(s, max(excl, carry));
    if (i < ni) { is[i] = (uint32_t)s2; ie[i] = (uint32_t)max(e, s2); }
    carry = max(carry, __shfl_sync(0xffffffffu, incl, 31));
  }
  __syncwarp();

  // (2) deltas sorted by site, stable: the last delta of a site in array order is the last of its run
  for (int i = lane; i < nd; i += 32) { dk0[i] = (uint32_t)P.delta_site[d0 + i]; dv0[i] = P.delta_to[d0 + i]; }
  __syncwarp();
  const bool dalt = warp_radix_sort(dk0, dv0, dk1, dv1, nd, P.site_bits, cnt, lane);
  const uint32_t* ds = dalt ? dk1 : dk0;
  const uint32_t* dt = dalt ? dv1 : dv0;

  // (3) the endpoints (position, +-c) of every mutation of A with c != 0
  if (lane == 0) s_n[warp] = 0;
  __syncwarp();
  int B = 0;
  for (int i = lane; i < nd; i += 32) {
    const int l = (int)ds[i];
    if (i + 1 < nd && (int)ds[i + 1] == l) continue;
    int lo = 0, hi = ni;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if ((int)is[mid] <= l) lo = mid + 1; else hi = mid; }
    if (lo > 0 && l < (int)ie[lo - 1]) continue;
    const int x = (int)dt[i];
    B += x != (int)P.ref[l];
    for (int j = P.site_off[l]; j < P.site_off[l + 1]; ++j) {
      const int4 m = __ldg(P.rec + j);
      const int c = (int)((m.z & 3) != x) - (int)((m.z >> 2) != x) - m.w;
      if (c) { const int q = atomicAdd(&s_n[warp], 2); ek0[q] = (uint32_t)m.x; ev0[q] = (uint32_t)c; ek0[q + 1] = (uint32_t)m.y; ev0[q + 1] = (uint32_t)-c; }
    }
  }
  constexpr int kLanePiece = 64;        // pieces with more mutations than this are spread over the warp
  for (int i = lane; i < ni; i += 32) {
    const int j0 = P.site_off[is[i]], j1 = P.site_off[ie[i]];
    if (j1 - j0 > kLanePiece) continue;
    for (int j = j0; j < j1; ++j) {
      const int4 m = __ldg(P.rec + j);
      if (m.w) { const int q = atomicAdd(&s_n[warp], 2); ek0[q] = (uint32_t)m.x; ev0[q] = (uint32_t)-m.w; ek0[q + 1] = (uint32_t)m.y; ev0[q + 1] = (uint32_t)m.w; }
    }
  }
  for (int i = 0; i < ni; ++i) {
    const int j0 = P.site_off[is[i]], j1 = P.site_off[ie[i]];
    if (j1 - j0 <= kLanePiece) continue;
    for (int j = j0 + lane; j < j1; j += 32) {
      const int4 m = __ldg(P.rec + j);
      if (m.w) { const int q = atomicAdd(&s_n[warp], 2); ek0[q] = (uint32_t)m.x; ev0[q] = (uint32_t)-m.w; ek0[q + 1] = (uint32_t)m.y; ev0[q + 1] = (uint32_t)m.w; }
    }
  }
  B = warp_sum(B);
  __syncwarp();
  const int n = s_n[warp];
  const bool ealt = warp_radix_sort(ek0, ev0, ek1, ev1, n, P.pos_bits, cnt, lane);
  const uint32_t* ks = ealt ? ek1 : ek0;
  const uint32_t* vs = ealt ? ev1 : ev0;

  // (4) sweep: piece j in [-1, n) is [pos_j, pos_{j+1}) (pos_{-1} = first region, pos_n = R) with correction = prefix of c up to j;
  // with a date limit only the regions with t_min < t_X count: the first K in t_min order
  const double tX = P.t_X ? P.t_X[k] : DBL_MAX;
  int K = P.R;
  if (P.tkey) {
    int lo = 0, hi = P.R;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (__ldg(P.tkey + mid) < tX) lo = mid + 1; else hi = mid; }
    K = lo;
  }
  const int start0 = P.can_change_root ? 0 : 1;
  int bv = INT_MAX, bc = 0, bl = 0, bm = 0;
  carry = 0;
  for (int b0 = -1; b0 < n; b0 += 32) {
    const int j = b0 + lane;
    const int c = (j >= 0 && j < n) ? (int)vs[j] : 0;
    const int corr = warp_scan_incl(c, lane) + carry;
    carry = __shfl_sync(0xffffffffu, corr, 31);
    if (j < n) {
      const int l = j < 0 ? start0 : max((int)ks[j], start0), r = j + 1 < n ? (int)ks[j + 1] : P.R;
      const int2 q = l < r ? place_query(P, K, l, r) : make_int2(INT_MAX, 0);
      if (q.y > 0) {                    // a piece without kept regions (only under a date limit) offers nothing
        const int v = q.x + corr;
        if (v < bv) { bv = v; bc = q.y; bl = l; bm = q.x; }
        else if (v == bv) bc += q.y;
      }
    }
  }
  const int best = warp_min(bv);
  const int count = warp_sum(bv == best ? bc : 0);
  const int first_l = warp_min(bv == best ? bl : INT_MAX);
  int first = -1;
  const unsigned owner = __ballot_sync(0xffffffffu, bv == best && bl == first_l && best != INT_MAX);
  if (owner) {
    const int ol = __ffs(owner) - 1;
    if (lane == ol) first = place_find_first(P, K, bl, bm);
    first = __shfl_sync(0xffffffffu, first, ol);
  }
  if (lane == 0) {
    dphy_placement o;
    o.min_muts = -1; o.num_best = 0; o.branch = -1; o.mut_idx = -1;
    if (first >= 0) {
      const dphy_candidate_region fr = place_region_record(P, first, tX);
      o.min_muts = B + best; o.num_best = count; o.branch = fr.branch; o.mut_idx = fr.mut_idx;
    }
    P.out[k] = o;
  }
  if (P.max_best <= 0) return;

  // (5) the first max_best regions attaining the minimum, in emission order: the pieces whose minimum hits it, leaf by leaf
  dphy_candidate_region* bo = P.best + (size_t)k * P.max_best;
  int emitted = 0;
  carry = 0;
  for (int b0 = -1; first >= 0 && b0 < n && emitted < P.max_best; b0 += 32) {
    const int j = b0 + lane;
    const int c = (j >= 0 && j < n) ? (int)vs[j] : 0;
    const int corr = warp_scan_incl(c, lane) + carry;
    carry = __shfl_sync(0xffffffffu, corr, 31);
    int l = 0, r = 0, hit = 0, m = 0;
    if (j < n) {
      l = j < 0 ? start0 : max((int)ks[j], start0); r = j + 1 < n ? (int)ks[j + 1] : P.R;
      if (l < r) { const int2 q = place_query(P, K, l, r); m = q.x; hit = q.y > 0 && q.x + corr == best ? q.y : 0; }
    }
    const int incl = warp_scan_incl(hit, lane);
    const int off = emitted + incl - hit;
    const int take = off < P.max_best ? min(hit, P.max_best - off) : 0;
    for (int t = 0; t < take; ++t) {
      const int p = place_find_first(P, K, l, m);
      dphy_candidate_region rr = place_region_record(P, p, tX);
      rr.min_muts = B + best;
      bo[off + t] = rr;
      l = p + 1;
    }
    emitted = min(P.max_best, emitted + __shfl_sync(0xffffffffu, incl, 31));
  }
  for (int t = emitted + lane; t < P.max_best; t += 32) {
    dphy_candidate_region u;
    u.branch = -1; u.mut_idx = 0; u.t_min = 0.0; u.t_max = 0.0; u.min_muts = 0; u.pad_ = 0; u.log_W_over_Wmax = 0.0; u.W_over_Wmax = 0.0;
    bo[t] = u;
  }
}

namespace {

// the per-tree index: built by the first placement on the tree, freed with the forest (dphy_forest_apply_rows swaps in a fresh forest,
// so a rebuilt tree gets a fresh index; dphy_forest_set_node_times changes no entry, the times are read when the records are made)
int ensure_place_index(dphy_ctx* ctx, dphy_forest* fo, int tree) {
  if (fo->place.size() != fo->trees.size()) fo->place.assign(fo->trees.size(), PlaceIndex{});
  PlaceIndex& X = fo->place[tree];
  if (X.seg) return DPHY_OK;
  const TreeDev& T = fo->trees[tree];
  const dphy_sites* si = fo->sites[T.sites_id];
  const int nb = T.node_base, N = T.num_nodes, L = si->L;
  int32_t h_mo[3];
  DPHY_CUDA(ctx, cudaMemcpyAsync(h_mo, fo->h.mut_off + nb, sizeof(int32_t) * 2, cudaMemcpyDeviceToHost, ctx->stream));
  DPHY_CUDA(ctx, cudaMemcpyAsync(h_mo + 2, fo->h.mut_off + nb + N, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DPHY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  const int64_t M = (int64_t)h_mo[2] - h_mo[0];
  const int64_t R = (int64_t)N + M - (h_mo[1] - h_mo[0]);
  if (R + 2 >= (int64_t)1 << 30) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "place: tree too large");
  int64_t P2 = 1;
  while (P2 < R) P2 <<= 1;
  // resident: site_off [L+1], rec [M], seg [2 P2]; temporaries (freed once built): fill [L], diff [R+2], scan tiles
  Slab res, work;
  const int b_so = res.reserve(sizeof(int32_t) * (L + 1)), b_rec = res.reserve(sizeof(int4) * std::max<int64_t>(M, 1));
  const int b_seg = res.reserve(sizeof(int2) * 2 * P2);
  const int b_fill = work.reserve(sizeof(int32_t) * L), b_diff = work.reserve(sizeof(int32_t) * (R + 2));
  const int b_tt = work.reserve(sizeof(int32_t) * ((std::max<int64_t>(L, R + 1) + 1) / 8192 + 2));
  DevBlock d(ctx->stream), tmp(ctx->stream);
  if (!d.alloc(res.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(place index)");
  if (!tmp.alloc(work.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(place index scratch)");
  int32_t* so = res.at<int32_t>(d.p, b_so); int4* rec = res.at<int4>(d.p, b_rec); int2* seg = res.at<int2>(d.p, b_seg);
  int32_t* fill = work.at<int32_t>(tmp.p, b_fill); int32_t* diff = work.at<int32_t>(tmp.p, b_diff); int32_t* tt = work.at<int32_t>(tmp.p, b_tt);
  // site_off, fill and diff start at zero
  int st = check_cuda(ctx, cudaMemsetAsync(d.p, 0, res.blocks[b_rec].off, ctx->stream), "place index memset");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaMemsetAsync(tmp.p, 0, work.blocks[b_tt].off, ctx->stream), "place index memset");
  if (st == DPHY_OK) {
    const int m0 = h_mo[0], Mi = (int)M;
    if (Mi > 0) place_site_hist_kernel<<<(Mi + 255) / 256, 256, 0, ctx->stream>>>(fo->h, m0, Mi, so);
    st = launch_scan_i32(ctx, so, L + 1, tt);
    if (st == DPHY_OK && Mi > 0)
      place_site_scatter_kernel<<<(Mi + 255) / 256, 256, 0, ctx->stream>>>(fo->h, nb, N, (int)R, m0, Mi, si->d_ref, so, fill, rec, diff);
    if (st == DPHY_OK) st = launch_scan_i32(ctx, diff, (int)R + 2, tt);
    if (st == DPHY_OK) {
      place_seg_leaves_kernel<<<(unsigned)((P2 + 255) / 256), 256, 0, ctx->stream>>>(diff, (int)R, (int)P2, seg);
      ctx->launches += 3;
      for (int64_t lo = P2 / 2; lo >= 1; lo /= 2) { place_seg_level_kernel<<<(unsigned)((lo + 255) / 256), 256, 0, ctx->stream>>>(seg, (int)lo); ++ctx->launches; }
      st = check_cuda(ctx, cudaGetLastError(), "place index kernels");
    }
  }
  std::vector<int32_t> h_so(L + 1);
  if (st == DPHY_OK) st = check_cuda(ctx, cudaMemcpyAsync(h_so.data(), so, sizeof(int32_t) * (L + 1), cudaMemcpyDeviceToHost, ctx->stream), "D2H");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "place index build");
  tmp.reset();
  if (st != DPHY_OK) return st;
  fo->allocs.push_back(d.release());
  fo->bytes += res.total;
  X.R = (int32_t)R; X.P2 = (int32_t)P2; X.L = L;
  X.site_off = so; X.rec = rec; X.seg = seg;
  X.h_site_off = std::move(h_so);
  return DPHY_OK;
}

// the largest t_min of the tree (a date limit above it drops no region), cached per times version
int place_max_key(dphy_ctx* ctx, dphy_forest* fo, int tree, uint64_t ver) {
  PlaceIndex& X = fo->place[tree];
  if (X.max_at == ver) return DPHY_OK;
  const TreeDev& T = fo->trees[tree];
  const size_t mark = ctx->arena.mark();
  unsigned long long* d_max = (unsigned long long*)ctx->arena.alloc(sizeof(unsigned long long));
  if (!d_max) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "arena exhausted (place)");
  unsigned long long h_max = 0;
  int st = check_cuda(ctx, cudaMemsetAsync(d_max, 0, sizeof(unsigned long long), ctx->stream), "place memset");
  if (st == DPHY_OK) {
    place_tkey_max_kernel<<<(T.num_nodes + 255) / 256, 256, 0, ctx->stream>>>(fo->h, T.node_base, T.num_nodes, d_max);
    ++ctx->launches;
    st = check_cuda(ctx, cudaGetLastError(), "place_tkey_max_kernel");
  }
  if (st == DPHY_OK) st = check_cuda(ctx, cudaMemcpyAsync(&h_max, d_max, sizeof(h_max), cudaMemcpyDeviceToHost, ctx->stream), "D2H");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "place max key");
  ctx->arena.release(mark);
  if (st != DPHY_OK) return st;
  const unsigned long long u = (h_max >> 63) ? h_max & ~(1ull << 63) : ~h_max;
  std::memcpy(&X.max_key, &u, sizeof(u));
  X.max_at = ver;
  return DPHY_OK;
}

// The dated part of the index (lc / pre: lg levels x P2 entries, 12 B each; tkey: 8 B per region).  Its block is allocated by the
// first build and reused by every rebuild (R and P2 do not depend on times).  Level by level from the root: the level's list (the
// regions of each node in t_min order; the root's is the sorted order itself) is scanned per node for (left-child count, min Hr,
// count), which gives the level's tables and, by a stable partition on the next bit of the region index, the next level's list.
int ensure_dated_index(dphy_ctx* ctx, dphy_forest* fo, int tree, uint64_t ver) {
  PlaceIndex& X = fo->place[tree];
  if (X.tkey && X.dated_at == ver) return DPHY_OK;
  const TreeDev& T = fo->trees[tree];
  const int R = X.R, P2 = X.P2;
  int lg = 0;
  while ((1 << lg) < P2) ++lg;
  size_t sort_bytes = 0, scan_bytes = 0;
  DPHY_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const double*)nullptr, (double*)nullptr, (const int32_t*)nullptr,
                                                 (int32_t*)nullptr, R, 0, 64, ctx->stream));
  DPHY_CUDA(ctx, cub::DeviceScan::InclusiveScanByKey(nullptr, scan_bytes, thrust::counting_iterator<int>(0), (const DatedAcc*)nullptr,
                                                     (DatedAcc*)nullptr, DatedComb{}, P2, SameNode{1}, ctx->stream));
  Slab res, work;
  const int b_tkey = res.reserve(sizeof(double) * R), b_lc = res.reserve(sizeof(int32_t) * (size_t)lg * P2);
  const int b_pre = res.reserve(sizeof(int2) * (size_t)lg * P2);
  // temporaries: unsorted keys, region indices, two level lists, scan input and output, CUB's storage
  const int b_key = work.reserve(sizeof(double) * R), b_idx = work.reserve(sizeof(int32_t) * R), b_l0 = work.reserve(sizeof(int32_t) * P2);
  const int b_l1 = work.reserve(sizeof(int32_t) * P2), b_vin = work.reserve(sizeof(DatedAcc) * P2), b_vout = work.reserve(sizeof(DatedAcc) * P2);
  const int b_cub = work.reserve(std::max(sort_bytes, scan_bytes));
  DevBlock d(ctx->stream), tmp(ctx->stream);
  const bool fresh = X.tkey == nullptr;
  if (fresh && !d.alloc(res.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(dated place index)");
  if (!tmp.alloc(work.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(dated place index scratch)");
  if (fresh) {
    fo->allocs.push_back(d.release());
    fo->bytes += res.total;
    void* base = fo->allocs.back();
    X.tkey = res.at<double>(base, b_tkey); X.lc = res.at<int32_t>(base, b_lc); X.pre = res.at<int2>(base, b_pre); X.lg = lg;
  }
  X.dated_at = ~0ull;                       // not valid until the build below has finished
  double* key = work.at<double>(tmp.p, b_key); int32_t* idx = work.at<int32_t>(tmp.p, b_idx);
  int32_t* list = work.at<int32_t>(tmp.p, b_l0); int32_t* next = work.at<int32_t>(tmp.p, b_l1);
  DatedAcc* vin = work.at<DatedAcc>(tmp.p, b_vin); DatedAcc* vout = work.at<DatedAcc>(tmp.p, b_vout); void* cub_tmp = work.at<char>(tmp.p, b_cub);
  place_tkey_kernel<<<(T.num_nodes + 255) / 256, 256, 0, ctx->stream>>>(fo->h, T.node_base, T.num_nodes, key, idx);
  if (P2 > R) place_pad_list_kernel<<<(P2 - R + 255) / 256, 256, 0, ctx->stream>>>(list, R, P2);
  // every CUB call below is counted as one launch
  cudaError_t ce = cub::DeviceRadixSort::SortPairs(cub_tmp, sort_bytes, (const double*)key, X.tkey, (const int32_t*)idx, list, R, 0, 64,
                                                   ctx->stream);
  ctx->launches += 3;
  const unsigned blocks = (unsigned)((P2 + 255) / 256);
  for (int lv = lg; lv >= 1 && ce == cudaSuccess; --lv) {
    place_dated_vals_kernel<<<blocks, 256, 0, ctx->stream>>>(list, X.seg, P2, lv, vin);
    ce = cub::DeviceScan::InclusiveScanByKey(cub_tmp, scan_bytes, thrust::counting_iterator<int>(0), (const DatedAcc*)vin, vout,
                                             DatedComb{}, P2, SameNode{lv}, ctx->stream);
    if (ce == cudaSuccess)
      place_dated_level_kernel<<<blocks, 256, 0, ctx->stream>>>(list, vout, P2, lv, X.lc + (size_t)(lv - 1) * P2,
                                                                 X.pre + (size_t)(lv - 1) * P2, next);
    std::swap(list, next);
    ctx->launches += 3;
  }
  int st = check_cuda(ctx, ce, "dated place index");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaGetLastError(), "dated place index kernels");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "dated place index build");
  tmp.reset();
  if (st == DPHY_OK) X.dated_at = ver;
  return st;
}

// dphy_forest_place_samples (t_X == nullptr, dated == false) and dphy_forest_place_dated_samples
int place_samples(dphy_ctx* ctx, dphy_forest* fo, int32_t tree, const dphy_sample_set* set, const double* t_X, bool dated,
                  int32_t can_change_root, int32_t max_best, dphy_placement* out, dphy_candidate_region* best) {
  if (!ctx || !fo || !set || max_best < 0 || set->num_samples < 0) return DPHY_ERR_INVALID_ARGUMENT;
  if (tree < 0 || tree >= fo->h.num_trees) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "place: tree index out of range");
  const int S = set->num_samples;
  if (S == 0) return DPHY_OK;
  if (!out || (max_best > 0 && !best)) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "place: output buffers missing");
  if (!set->delta_off || !set->miss_off) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "place: offset arrays missing");
  // ---- validation (the rules of a DPHY_SPR_X_REL_REF request), before anything is written ----
  const int32_t* dof = set->delta_off; const int32_t* mof = set->miss_off;
  if (dof[0] < 0 || mof[0] < 0) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "place: negative offsets");
  for (int k = 0; k < S; ++k)
    if (dof[k + 1] < dof[k] || mof[k + 1] < mof[k]) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "place: offsets not monotone");
  const int64_t D = (int64_t)dof[S] - dof[0], I = (int64_t)mof[S] - mof[0];
  if ((D > 0 && (!set->delta_site || !set->delta_to)) || (I > 0 && (!set->miss_start || !set->miss_end)))
    return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "place: sample arrays missing");
  const TreeDev& T = fo->trees[tree];
  const int L = fo->sites[T.sites_id]->L;
  for (int64_t i = dof[0]; i < dof[S]; ++i)
    if (set->delta_site[i] < 0 || set->delta_site[i] >= L || set->delta_to[i] > 3) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "place: delta out of range");
  for (int64_t i = mof[0]; i < mof[S]; ++i)
    if (set->miss_start[i] < 0 || set->miss_end[i] > L || set->miss_start[i] >= set->miss_end[i])
      return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "place: missing interval out of range");
  if (dated && !t_X) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "place: t_X missing");
  if (dated)
    for (int k = 0; k < S; ++k)
      if (std::isnan(t_X[k])) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "place: t_X is NaN");
  cudaSetDevice(ctx->device);
  int st = ensure_place_index(ctx, fo, tree);
  if (st != DPHY_OK) return st;
  const PlaceIndex& X = fo->place[tree];
  // the dated part is needed once some sample drops a region (t_X <= the largest t_min); a current one is used as it is
  bool use_dated = false;
  if (dated) {
    const uint64_t ver = fo->tree_times_version(tree);
    use_dated = X.tkey && X.dated_at == ver;
    if (!use_dated) {
      st = place_max_key(ctx, fo, tree, ver);
      if (st != DPHY_OK) return st;
      for (int k = 0; k < S && !use_dated; ++k) use_dated = t_X[k] <= X.max_key;
      if (use_dated) st = ensure_dated_index(ctx, fo, tree, ver);
      if (st != DPHY_OK) return st;
    }
  }
  // ---- scratch per sample: endpoint pairs (2 per mutation of A, bounded by the site table's runs), delta and interval pairs; each
  // ping-ponged by the radix sort: 4 words per pair ----
  const int32_t* so = X.h_site_off.data();
  std::vector<int64_t> scr(S + 1, 0);
  for (int k = 0; k < S; ++k) {
    int64_t a = 0;
    for (int i = dof[k]; i < dof[k + 1]; ++i) a += so[set->delta_site[i] + 1] - so[set->delta_site[i]];
    for (int i = mof[k]; i < mof[k + 1]; ++i) a += so[set->miss_end[i]] - so[set->miss_start[i]];
    if (2 * a > INT_MAX) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "place: sample too large");
    scr[k + 1] = scr[k] + 4 * (2 * a + (dof[k + 1] - dof[k]) + (mof[k + 1] - mof[k]));
  }
  // samples go in batches of at most kBudget scratch words (at least one sample per batch)
  constexpr int64_t kBudget = (int64_t)64 << 20;
  std::vector<int> cuts{0};
  int64_t max_words = 1;
  for (int k = 0; k < S; ++k) {
    if (k > cuts.back() && scr[k + 1] - scr[cuts.back()] > kBudget) cuts.push_back(k);
    max_words = std::max(max_words, scr[k + 1] - scr[cuts.back()]);
  }
  cuts.push_back(S);
  // ---- inputs through the pinned slab; outputs back through it ----
  // [inputs | outputs] cross through the pinned slab, the per-sample scratch stays on the device
  Slab slab;
  const int b_doff = slab.reserve(4 * (size_t)(S + 1)), b_moff = slab.reserve(4 * (size_t)(S + 1)), b_ds = slab.reserve(4 * (size_t)D);
  const int b_dt = slab.reserve((size_t)D), b_ms = slab.reserve(4 * (size_t)I), b_me = slab.reserve(4 * (size_t)I);
  const int b_scr = slab.reserve(8 * (size_t)(S + 1)), b_tx = dated ? slab.reserve(8 * (size_t)S) : -1;
  const size_t in_bytes = slab.total;
  const int b_out = slab.reserve(sizeof(dphy_placement) * (size_t)S), b_best = slab.reserve(sizeof(dphy_candidate_region) * (size_t)S * max_best);
  const size_t io_bytes = slab.total;
  const int b_scratch = slab.reserve(4 * (size_t)max_words);
  DevBlock blk(ctx->stream);
  if (!blk.alloc(slab.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(place)");
  char* d = blk.p;
  PinnedStage pin(ctx, io_bytes);
  if (pin.status != DPHY_OK) return pin.status;
  char* h = pin.p;
  int32_t* h_doff = slab.at<int32_t>(h, b_doff); int32_t* h_moff = slab.at<int32_t>(h, b_moff);
  for (int k = 0; k <= S; ++k) { h_doff[k] = dof[k] - dof[0]; h_moff[k] = mof[k] - mof[0]; }
  if (D) { std::memcpy(slab.at<char>(h, b_ds), set->delta_site + dof[0], 4 * D); std::memcpy(slab.at<char>(h, b_dt), set->delta_to + dof[0], D); }
  if (I) { std::memcpy(slab.at<char>(h, b_ms), set->miss_start + mof[0], 4 * I); std::memcpy(slab.at<char>(h, b_me), set->miss_end + mof[0], 4 * I); }
  std::memcpy(slab.at<char>(h, b_scr), scr.data(), 8 * (size_t)(S + 1));
  if (dated) std::memcpy(slab.at<char>(h, b_tx), t_X, 8 * (size_t)S);
  cudaError_t ce = cudaMemcpyAsync(d, h, in_bytes, cudaMemcpyHostToDevice, ctx->stream);
  PlaceParams P;
  std::memset(&P, 0, sizeof(P));
  P.f = fo->h; P.nb = T.node_base; P.N = T.num_nodes; P.R = X.R; P.P2 = X.P2; P.L = L;
  P.site_bits = bits_for(L); P.pos_bits = bits_for(X.R); P.can_change_root = can_change_root != 0; P.max_best = max_best;
  P.site_off = X.site_off; P.rec = X.rec; P.seg = X.seg; P.ref = fo->sites[T.sites_id]->d_ref;
  if (dated) P.t_X = slab.at<const double>(d, b_tx);
  if (use_dated) { P.tkey = X.tkey; P.lc = X.lc; P.pre = X.pre; P.lg = X.lg; }
  P.delta_off = slab.at<const int32_t>(d, b_doff); P.delta_site = slab.at<const int32_t>(d, b_ds); P.delta_to = slab.at<const uint8_t>(d, b_dt);
  P.miss_off = slab.at<const int32_t>(d, b_moff); P.miss_start = slab.at<const int32_t>(d, b_ms); P.miss_end = slab.at<const int32_t>(d, b_me);
  P.scr_off = slab.at<const int64_t>(d, b_scr); P.scratch = slab.at<uint32_t>(d, b_scratch);
  P.out = slab.at<dphy_placement>(d, b_out); P.best = slab.at<dphy_candidate_region>(d, b_best);
  for (size_t c = 0; c + 1 < cuts.size() && ce == cudaSuccess; ++c) {
    P.s0 = cuts[c]; P.s1 = cuts[c + 1];
    place_samples_kernel<<<(P.s1 - P.s0 + kPlaceWarps - 1) / kPlaceWarps, kPlaceWarps * 32, 0, ctx->stream>>>(P);
    ++ctx->launches;
    ce = cudaGetLastError();
  }
  const size_t out_at = slab.blocks[b_out].off;
  if (ce == cudaSuccess) ce = cudaMemcpyAsync(h + out_at, d + out_at, io_bytes - out_at, cudaMemcpyDeviceToHost, ctx->stream);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
  blk.reset();
  if (ce != cudaSuccess) return check_cuda(ctx, ce, "place samples");
  std::memcpy(out, slab.at<char>(h, b_out), sizeof(dphy_placement) * (size_t)S);
  if (max_best > 0) std::memcpy(best, slab.at<char>(h, b_best), sizeof(dphy_candidate_region) * (size_t)S * max_best);
  return DPHY_OK;
}
}  // namespace

}  // namespace dphy

using namespace dphy;

extern "C" {

int dphy_forest_place_samples(dphy_ctx* ctx, dphy_forest* fo, int32_t tree, const dphy_sample_set* set, int32_t can_change_root,
                              int32_t max_best, dphy_placement* out, dphy_candidate_region* best) {
  return place_samples(ctx, fo, tree, set, nullptr, false, can_change_root, max_best, out, best);
}

int dphy_forest_place_dated_samples(dphy_ctx* ctx, dphy_forest* fo, int32_t tree, const dphy_sample_set* set, const double* t_X,
                                    int32_t can_change_root, int32_t max_best, dphy_placement* out, dphy_candidate_region* best) {
  return place_samples(ctx, fo, tree, set, t_X, true, can_change_root, max_best, out, best);
}

}  // extern "C"
