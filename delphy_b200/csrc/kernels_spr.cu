// kernels_spr.cu -- batched SPR regraft studies on the device (sm_100a).
//
// Replaces, for a batch of studies in one pass over the forest:
//   reconstruct_missing_sites_at / view_of_sequence_at      core/phylo_tree_calc.cpp:19-56   (X's state + missing set)
//   Spr_study_builder::seed_fill_from (restricted DFS)       core/spr_study.cpp:9-128
//   Spr_study_builder::account_for_Xs_detachment             core/spr_study.cpp:130-209
//   Spr_study_builder::remove_regions_in_Xs_future           core/spr_study.cpp:211-224
//   Spr_study::Spr_study (region weights, max, exp, sum)     core/spr_study.cpp:226-385
//   Spr_study::pick_nexus_region / find_region               core/spr_study.cpp:404-422, :474-484
//
// Data-parallel restatement (SURVEY.md section 8a, row a12).  The reference walks the tree keeping a hash map of site
// deltas to X and reports min_muts = |map| per region.  Equivalently, with x_l = X's state and the per-mutation
// potential d(m) = [m.to != x_l] - [m.from != x_l] (0 where l is missing at X), min_muts(region) =
// min_muts(start) + H(region) - H(start) where H is the sum of d over the root->region path: one integer tree
// prefix sum.  The scope test (max_muts_from_start) is the path length in counted mutations, C(start->region) =
// C(start) + C(region) - 2 C(junction).  The DFS emission order is the pre-order of the region tree re-rooted at the
// start region; since nodes are stored in DFS order (children[1] first, exactly the order the builder's LIFO work
// stack produces), the output is a concatenation of O(depth) device-order segments whose bases come from one
// prefix sum of per-node kept-region counts, so every region's output index is computed independently.
#include "dphy_internal.h"
#include "device_utils.cuh"

#include <cooperative_groups.h>

#include <cfloat>
#include <climits>
#include <cmath>
#include <cstddef>
#include <cstring>
#include <memory>
#include <math_constants.h>
#include <new>
#include <vector>

namespace dphy {

// SprStudy::error: set on the device by the kernel named, turned into a status and a message by spr_fetch
enum SprError : int32_t {
  kSprErrXNoParent = 1,           // spr_init_kernel
  kSprErrStartMutIdx = 2,         // spr_init_kernel
  kSprErrStartInXSubtree = 3,     // spr_init_kernel
  kSprErrPathMuts = 4,            // spr_xtab_kernel: the root path's mutation ordinals must fit 28 bits
  kSprErrFrontierCap = 5,         // spr_frontier_kernel
  kSprErrHmixCap = 6,             // spr_g2_bases_kernel
};

struct SprStudy {
  // ---- inputs (host) ----
  int32_t tree, X, start_branch, start_mut_idx, init_min_muts, limit, can_change_root, n_x_deltas, n_x_missing;
  int32_t x_mode;          // DPHY_SPR_X_*: where X's state and missing set come from
  double t_X, lambda_X, f, t_max_tip;
  // slab offsets in bytes
  int64_t off_xtab, off_xkey, off_path, off_xpath, off_H, off_C, off_KB, off_seg, off_regions, off_xd_site, off_xd_to, off_xm_start,
      off_xm_end, off_part, off_pae, off_lw, off_tj, off_nw;
  int32_t region_cap, path_cap;
  // ---- derived (spr_setup_kernel) ----
  int32_t node_base, num_nodes, num_tiles, L;
  int32_t posX, posP, posS, nP, nS, P_is_root;
  int32_t pos0, k0, n0, root_pos;
  int32_t path_len, xpath_len;
  int32_t num_missing, error;
  int32_t C0, H0;          // counted-mutation depth / Hamming potential at the start region (set once H and C are scanned)
  int32_t scanned, pad2;   // bit 0: tile prefixes of H and C are final; bit 1: of the kept-region counts
  double mu;
  // ---- outputs ----
  int32_t total_regions, pad1;
  unsigned long long max_key;
  double log_Wmax, sum_W;
  // ---- layout of the tree prefix sums H / KB (and of their per-tile aggregates) ----
  // per-study path: one int per node (h_stride 1), tiles of kTile nodes (tile_shift 8);
  // grouped studies (h_stride 32) read H / KB off their group's event rows / keep masks instead (g2 fields below)
  int32_t h_stride, tile_shift, num_htiles, weights_fused;
  // event-scan grouped path (kernels_spr_group2.cuh): lane of the study inside its group and the group's tables (0 => not used)
  int32_t g2, g2_lane, g2_mut_base, g2_num_templates;
  int64_t off_g2S, off_g2aggS, off_g2mask, off_g2aggK, off_hang, off_hmix;
  int32_t hmix_cap, pad3;
};

// Device-side form of a candidate region: the reference's 48-byte Candidate_region (core/spr_study.h:17-32) split into a 32-byte
// head written by the emit kernel and a 16-byte (log_W_over_Wmax, W_over_Wmax) tail written by the normalisation kernel, each in
// its own array, so that both kernels store whole 32-byte sectors (a 16-byte store into a 48-byte record costs a DRAM
// read-modify-write: ncu showed 375 MB read for 78 MB of useful input).  dphy_spr_batch_get_regions interleaves them on the way out.
struct alignas(32) RegionHead { int32_t branch, mut_idx; double t_min, t_max; int32_t min_muts, pad; };
static_assert(sizeof(RegionHead) == 32, "RegionHead must be 32 bytes");

constexpr int kSegStride = 6;     // ints per path node: baseA, baseOwnDown, baseSub, baseUp, cntUp, sibpos
constexpr int kNormBlocks = 64;   // blocks per study in the normalisation pass (fixed => deterministic sum)

struct SprBatchDev {
  SprStudy* studies;
  char* slab;
  int32_t* tile_agg;      // [S][max_tiles + 1][3]: per-tile totals of (H, C, kept regions), then their exclusive prefixes
  uint32_t* tile_flag;    // unused
  uint32_t* ticket;       // [S][4]
  int32_t num_studies, max_tiles;
  // study-independent tables of the forest for the event-scan path (built once per forest, dphy_forest::d_spr_*)
  const int32_t* g2_eopen;     // [num_nodes]  tree-local index of the event at which the node opens
  const int32_t* g2_tnode;     // [num_nodes + total mutations]  device position of the node of every region template
  const int32_t* g2_ev;        // [2 * total mutations]  tree-local mutation index | exit << 31, in event order
  const int32_t* g2_mut_off;   // == ForestDev::mut_off
};

__device__ __forceinline__ unsigned long long f64_order_key(double d) {
  unsigned long long b = (unsigned long long)__double_as_longlong(d);
  return (b & 0x8000000000000000ULL) ? ~b : (b | 0x8000000000000000ULL);
}
__device__ __forceinline__ double f64_from_order_key(unsigned long long k) {
  unsigned long long b = (k & 0x8000000000000000ULL) ? (k & 0x7FFFFFFFFFFFFFFFULL) : ~k;
  return __longlong_as_double((long long)b);
}

// ---- Q(a,x): regularized upper incomplete gamma (series / continued fraction), as in safe_gamma_math.h:46-51 -----------
__device__ __noinline__ double dev_gamma_q(double a, double x) {
  if (x <= 0.0) return 1.0;
  if (isinf(x)) return 0.0;
  if (x < a + 1.0) {
    double sum = 1.0, term = 1.0, ap = a;
    for (int n = 0; n < 100000; ++n) { ap += 1.0; term *= x / ap; sum += term; if (fabs(term) < fabs(sum) * 1e-17) break; }
    double p = sum * exp(a * log(x) - x - lgamma(a + 1.0));
    double q = 1.0 - p;
    return q < 0.0 ? 0.0 : (q > 1.0 ? 1.0 : q);
  }
  const double tiny = 1e-300;
  double b = x + 1.0 - a, c = 1.0 / tiny, d = 1.0 / b, h = d;
  for (int i = 1; i < 100000; ++i) {
    const double an = -(double)i * ((double)i - a);
    b += 2.0;
    d = an * d + b; if (fabs(d) < tiny) d = tiny;
    c = b + an / c; if (fabs(c) < tiny) c = tiny;
    d = 1.0 / d;
    const double del = d * c;
    h *= del;
    if (fabs(del - 1.0) < 1e-16) break;
  }
  double q = exp(a * log(x) - x - lgamma(a)) * h;
  return q < 0.0 ? 0.0 : (q > 1.0 ? 1.0 : q);
}

// ---- (1) per-study setup: node positions, root paths, X's state table -------------------------------------------------------
// Everything is grid-parallel: no thread ever chases parent pointers.  In DFS pre-order the ancestors of q are exactly
// the positions p <= q with p + subtree_size[p] > q, and the ancestor at depth d goes to slot depth[q] - d of the path,
// so both root paths are built by one coalesced sweep over subtree_size (spr_paths_kernel, grid = position chunks x studies).
// X's sequence is the reference sequence overlaid with the LAST mutation per site on the root->X path: every path mutation
// posts (ordinal << 2 | to) with an atomicMax on a per-site key, ordinals coming from a block scan of the per-branch list
// lengths in root->X order (spr_xtab_kernel, one CTA per study).
constexpr int kSetupThreads = 1024;

// (a) spr_init_kernel (one CTA per tree of the batch): per study -- node positions, P / S, the derived fields, and the study's two
//     path TARGETS (its start node and X); then the tree's targets sorted by position (rank by counting: a batch has a few
//     hundred);  (b) spr_paths_kernel: ONE sweep over the tree for all its studies -- position p is an ancestor-or-self of
//     target t iff p <= t < p + subtree_size[p], i.e. the targets of p are a contiguous run of the sorted list, found by two binary
//     searches in shared memory; cost per position independent of the number of studies (the per-study sweep it replaces issued
//     26 M instructions for 128 studies of a 100k-tip tree).
struct SprPathTree { int32_t tree, first, count, pad; };     // studies order[first .. first + count) address this tree

// Per path target (sorted by position): where its ancestors go.  base = (length of the study's path to that target) - 1.
struct alignas(16) SprPathTarget { int32_t pos, base; uint32_t off_lo, off_hi; };      // off = slab offset of path[] (start) / xpath[] (X)
struct alignas(8) SprPathTargetAux { uint32_t pae_lo, pae_hi; };                        // slab offset of pae[] (start targets), 0 for X

__global__ void __launch_bounds__(256) spr_init_kernel(ForestDev f, SprBatchDev B, const SprPathTree* __restrict__ ptrees,
                                                       const int32_t* __restrict__ order, int32_t* __restrict__ traw,
                                                       SprPathTarget* __restrict__ tgt, SprPathTargetAux* __restrict__ aux) {
  const SprPathTree PT = ptrees[blockIdx.x];
  for (int w = threadIdx.x; w < PT.count; w += 256) {
    const int i = order[PT.first + w];
    SprStudy& S = B.studies[i];
    const TreeDev T = f.trees[S.tree];
    const int pos0 = T.node_base + f.pos_of_node[T.node_base + S.start_branch];
    const int posX = S.X >= 0 ? T.node_base + f.pos_of_node[T.node_base + S.X] : -1;
    const int dep0 = f.depth[pos0], depX = posX >= 0 ? f.depth[posX] : -1;
    S.node_base = T.node_base; S.num_nodes = T.num_nodes; S.num_tiles = T.num_tiles; S.L = f.sites[T.sites_id].L;
    S.root_pos = T.node_base; S.error = 0; S.scanned = 0; S.C0 = 0; S.H0 = 0;
    S.num_missing = 0;
    S.total_regions = 0; S.max_key = 0ULL; S.log_Wmax = 0.0; S.sum_W = 0.0;
    int posP = -1, posS = -1, nP = 0, nS = 0, Proot = 0;
    if (posX >= 0) {
      posP = f.parent_pos[posX];
      if (posP < 0) { S.error = kSprErrXNoParent; posP = posX; }
      const int c1 = posP + 1, c0 = posP + 1 + f.subtree_size[posP + 1];
      posS = (posX == c1) ? c0 : c1;
      nP = f.mut_off[posP + 1] - f.mut_off[posP];
      nS = f.mut_off[posS + 1] - f.mut_off[posS];
      Proot = f.parent_pos[posP] < 0;
    }
    S.posX = posX; S.posP = posP; S.posS = posS; S.nP = nP; S.nS = nS; S.P_is_root = Proot;
    S.pos0 = pos0; S.k0 = S.start_mut_idx; S.n0 = f.mut_off[pos0 + 1] - f.mut_off[pos0];
    if (S.k0 < 0 || S.k0 > S.n0 || (pos0 == T.node_base && S.k0 != S.n0)) S.error = kSprErrStartMutIdx;
    if (posX >= 0 && pos0 >= posX && pos0 < posX + f.subtree_size[posX]) S.error = kSprErrStartInXSubtree;   // start inside X's subtree
    S.path_len = min(dep0 + 1, S.path_cap);
    S.xpath_len = posX >= 0 ? min(depX + 1, S.path_cap) : 0;
    traw[2 * (PT.first + w)] = pos0; traw[2 * (PT.first + w) + 1] = posX >= 0 ? posX : INT_MAX;
  }
  __syncthreads();
  // the tree's targets sorted by position (rank by counting: a batch has a few hundred)
  const int T2 = 2 * PT.count;
  const int32_t* tr = traw + 2 * PT.first;
  for (int a = threadIdx.x; a < T2; a += 256) {
    const int pa = tr[a];
    int rank = 0;
    for (int b2 = 0; b2 < T2; ++b2) { const int pb = tr[b2]; rank += (pb < pa || (pb == pa && b2 < a)) ? 1 : 0; }
    const SprStudy& S = B.studies[order[PT.first + (a >> 1)]];
    SprPathTarget t; SprPathTargetAux x;
    t.pos = pa;
    if (a & 1) { t.base = S.xpath_len - 1; t.off_lo = (uint32_t)S.off_xpath; t.off_hi = (uint32_t)((unsigned long long)S.off_xpath >> 32); x.pae_lo = 0u; x.pae_hi = 0u; }
    else {
      t.base = S.path_len - 1; t.off_lo = (uint32_t)S.off_path; t.off_hi = (uint32_t)((unsigned long long)S.off_path >> 32);
      x.pae_lo = (uint32_t)S.off_pae; x.pae_hi = (uint32_t)((unsigned long long)S.off_pae >> 32);
    }
    tgt[2 * PT.first + rank] = t; aux[2 * PT.first + rank] = x;
  }
}

constexpr int kPathTargetsSmem = 1024;      // targets per slice of the sweep (512 studies of one tree)
__global__ void __launch_bounds__(kSetupThreads) spr_paths_kernel(ForestDev f, SprBatchDev B, const SprPathTree* __restrict__ ptrees,
                                                                  const SprPathTarget* __restrict__ tgt, const SprPathTargetAux* __restrict__ aux) {
  __shared__ SprPathTarget s_t[kPathTargetsSmem];
  __shared__ SprPathTargetAux s_x[kPathTargetsSmem];
  __shared__ int s_start[kSetupThreads + 1], s_lo[kSetupThreads], s_end[kSetupThreads], s_dep[kSetupThreads];
  __shared__ int s_ws[kSetupThreads / 32];
  const SprPathTree PT = ptrees[blockIdx.y];
  const TreeDev T = f.trees[PT.tree];
  const int tid = threadIdx.x;
  const int p = T.node_base + blockIdx.x * kSetupThreads + tid;
  if ((long long)blockIdx.x * kSetupThreads >= T.num_nodes) return;
  const bool in_tree = p < T.node_base + T.num_nodes;
  const int end = in_tree ? p + f.subtree_size[p] : 0;
  const int dep = in_tree ? f.depth[p] : 0;
  const int T2 = 2 * PT.count;
  for (int t0 = 0; t0 < T2; t0 += kPathTargetsSmem) {          // (one slice unless a tree has more than 512 studies in the batch)
    const int nt = min(kPathTargetsSmem, T2 - t0);
    __syncthreads();
    for (int i = tid; i < nt; i += kSetupThreads) { s_t[i] = tgt[2 * PT.first + t0 + i]; s_x[i] = aux[2 * PT.first + t0 + i]; }
    __syncthreads();
    // the targets below this node: a run [lo, lo + cnt) of the sorted list
    int lo = 0, cnt = 0;
    if (in_tree) {
      int hi = nt;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (s_t[mid].pos < p) lo = mid + 1; else hi = mid; }
      int l2 = lo; hi = nt;
      while (l2 < hi) { const int mid = (l2 + hi) >> 1; if (s_t[mid].pos < end) l2 = mid + 1; else hi = mid; }
      cnt = l2 - lo;
    }
    // (node, target) pairs spread evenly over the CTA: the nodes near the root are above EVERY target, one thread each would
    // serialise hundreds of stores; everything a pair needs is in shared memory, so a pair is a search and one or two stores
    int total;
    const int incl = block_scan_incl<int, kSetupThreads>(cnt, s_ws, &total);
    s_start[tid] = incl - cnt; s_lo[tid] = lo; s_end[tid] = end; s_dep[tid] = dep;
    if (tid == 0) s_start[kSetupThreads] = total;
    __syncthreads();
    for (int w = tid; w < total; w += kSetupThreads) {
      int a = 0, bnd = kSetupThreads - 1;                        // last node whose run starts at or before pair w
      while (a < bnd) { const int mid = (a + bnd + 1) >> 1; if (s_start[mid] <= w) a = mid; else bnd = mid - 1; }
      const int node = T.node_base + blockIdx.x * kSetupThreads + a;
      const int ti = s_lo[a] + (w - s_start[a]);
      const SprPathTarget t = s_t[ti];
      const int slot = t.base - s_dep[a];
      if (slot >= 0) {
        ((int32_t*)(B.slab + (((unsigned long long)t.off_hi << 32) | t.off_lo)))[slot] = node;
        const SprPathTargetAux x = s_x[ti];
        const unsigned long long po = ((unsigned long long)x.pae_hi << 32) | x.pae_lo;
        if (po) ((int2*)(B.slab + po))[slot] = make_int2(node, s_end[a]);     // classify() searches these nested [start, end) ranges
      }
    }
  }
}

constexpr int kXtabSlices = 2;     // CTAs per study: each owns a contiguous slice of the sites
__global__ void __launch_bounds__(kSetupThreads) spr_xtab_kernel(ForestDev f, SprBatchDev B) {
  __shared__ int s_ws[kSetupThreads / 32];
  __shared__ int s_carry;
  SprStudy& S = B.studies[blockIdx.y];
  const int tid = threadIdx.x;
  const TreeDev T = f.trees[S.tree];
  const SitesDev& Si = f.sites[T.sites_id];
  const int L = Si.L;
  const int X = S.X;
  // this CTA's sites: [l0, l1), a multiple of 128 long so that no two CTAs share a line of xtab / xkey
  const int per = ((L + kXtabSlices - 1) / kXtabSlices + 127) & ~127;
  const int l0 = min((int)blockIdx.x * per, L), l1 = min(l0 + per, L);
  uint8_t* xtab = (uint8_t*)(B.slab + S.off_xtab);
  uint32_t* xkey = (uint32_t*)(B.slab + S.off_xkey);
  for (int l = l0 + tid; l < l1; l += kSetupThreads) { xtab[l] = Si.ref[l]; xkey[l] = 0u; }
  if (tid == 0) s_carry = 0;
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31;
  // The state table is the reference sequence overlaid with the LAST mutation per site along a root-ward path, then with the
  // caller's deltas.  Which path:  FROM_TREE -> root..X (view_of_sequence_at(X));  REL_START -> root..start region (the state the
  // builder's cur_to_X_deltas are relative to, core/spr_study.cpp:9-24), start branch truncated to its first k0 mutations;
  // REL_REF -> none (deltas are relative to the reference sequence).
  const bool from_tree = S.x_mode == DPHY_SPR_X_FROM_TREE && X >= 0;
  const bool rel_start = S.x_mode == DPHY_SPR_X_REL_START;
  const int32_t* xpath = from_tree ? (const int32_t*)(B.slab + S.off_xpath) : (const int32_t*)(B.slab + S.off_path);
  const int xpath_len = from_tree ? S.xpath_len : (rel_start ? S.path_len : 0);
  if (from_tree) {
    // missing_at_X = union of the missation intervals on the X->root path (disjoint along a path by invariant).  The path nodes'
    // interval ranges are gathered by all threads at once and scanned, then the warps take the INTERVALS in turn (owner by binary
    // search in shared memory), lanes striding over the sites that fall into this CTA's slice: one round of dependent loads instead
    // of one per path node (a warp per path node was a chain of ~13 x 4 load latencies, most of this kernel's 38 us)
    __shared__ int s_ist[kSetupThreads + 1], s_io0[kSetupThreads];
    for (int j0 = 0; j0 < xpath_len; j0 += kSetupThreads) {
      const int j = j0 + tid;
      int o0 = 0, c = 0;
      if (j < xpath_len) { const int a = xpath[j]; o0 = f.miss_off[a]; c = f.miss_off[a + 1] - o0; }
      int tot;
      const int incl = block_scan_incl<int, kSetupThreads>(c, s_ws, &tot);
      s_ist[tid] = incl - c; s_io0[tid] = o0;
      if (tid == 0) s_ist[kSetupThreads] = tot;
      __syncthreads();
      for (int w = warp; w < tot; w += kSetupThreads / 32) {
        int a = 0, b = kSetupThreads - 1;                      // last path node whose intervals start at or before w
        while (a < b) { const int mid = (a + b + 1) >> 1; if (s_ist[mid] <= w) a = mid; else b = mid - 1; }
        const int2 se = f.miss_se[s_io0[a] + (w - s_ist[a])];
        for (int l = max(se.x, l0) + lane; l < min(se.y, l1); l += 32) xtab[l] |= 4;
      }
      __syncthreads();
    }
  } else {
    const int32_t* ms = (const int32_t*)(B.slab + S.off_xm_start);
    const int32_t* me = (const int32_t*)(B.slab + S.off_xm_end);
    for (int i = warp; i < S.n_x_missing; i += kSetupThreads / 32)
      for (int l = max(ms[i], l0) + lane; l < min(me[i], l1); l += 32) xtab[l] |= 4;
  }
  // last mutation per site on the path: every path mutation posts (ordinal << 2 | to) with an atomicMax on a per-site key
  // (every CTA walks the whole path -- it is short -- and posts the mutations of its own sites)
  for (int j0 = 0; j0 < xpath_len; j0 += kSetupThreads) {
    const int j = j0 + tid;                                   // j counts from the ROOT end of the path
    const int a = j < xpath_len ? xpath[xpath_len - 1 - j] : -1;
    const int mo = a >= 0 ? f.mut_off[a] : 0;
    int cnt = a >= 0 ? f.mut_off[a + 1] - mo : 0;
    if (rel_start && j == xpath_len - 1 && a != S.root_pos) cnt = min(cnt, S.start_mut_idx);   // region (start, k0): k0 mutations crossed
    int tot;
    const int incl = block_scan_incl<int, kSetupThreads>(cnt, s_ws, &tot);
    const int base = s_carry + incl - cnt;
    if (base + cnt >= (1 << 28)) S.error = kSprErrPathMuts;
    for (int i = 0; i < cnt; ++i) {
      const int site = f.mut_site[mo + i];
      if (site >= l0 && site < l1) atomicMax(xkey + site, ((uint32_t)(base + i + 1) << 2) | (uint32_t)(f.mut_code[mo + i] & 3));
    }
    __syncthreads();
    if (tid == 0) s_carry += tot;
    __syncthreads();
  }
  if (!from_tree) {
    const int32_t* ds = (const int32_t*)(B.slab + S.off_xd_site);
    const uint8_t* dt = (const uint8_t*)(B.slab + S.off_xd_to);
    const int base = s_carry;
    for (int i = tid; i < S.n_x_deltas; i += kSetupThreads) {
      const int site = ds[i];
      if (site >= l0 && site < l1) atomicMax(xkey + site, ((uint32_t)(base + i + 1) << 2) | (uint32_t)(dt[i] & 3));
    }
  }
  __syncthreads();
  int cnt = 0;
  for (int l = l0 + tid; l < l1; l += kSetupThreads) {
    const uint32_t k = __ldcg(xkey + l);
    uint8_t x = xtab[l];
    if (k) { x = (uint8_t)((x & 4) | (k & 3)); xtab[l] = x; }
    cnt += (x >> 2) & 1;
  }
  cnt = block_sum<int, kSetupThreads>(cnt, s_ws);
  if (tid == 0 && cnt) atomicAdd(&S.num_missing, cnt);      // zeroed by spr_paths_kernel; Spr_study::mu is set by spr_segments_kernel
}

// ---- shared device helpers ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mut_dc(const uint8_t* __restrict__ xtab, int site, int ft, int& dH, int& c) {
  const int xt = xtab[site];
  if (xt & 4) { dH = 0; c = 0; return; }
  const int x = xt & 3, from = ft >> 2, to = ft & 3;
  dH = (int)(to != x) - (int)(from != x);
  c = 1;
}

__device__ __forceinline__ void node_dc(const ForestDev& f, const uint8_t* __restrict__ xtab, int p, int& dH, int& dC) {
  dH = 0; dC = 0;
  for (int i = f.mut_off[p]; i < f.mut_off[p + 1]; ++i) {
    int h, c;
    mut_dc(xtab, f.mut_site[i], f.mut_code[i] & 15, h, c);
    dH += h; dC += c;
  }
}

// remove_regions_in_Xs_future (core/spr_study.cpp:211-224) drops every region that starts at or after t_X.  Every region of
// branch p starts at or after t[parent(p)], and so does everything below p: if t[parent(p)] >= t_X the branch and its whole
// subtree -- a contiguous range of positions -- contribute nothing, so the kernels neither walk their mutation lists nor give
// them output slots.  Exceptions: S and P (their regions are relabelled by account_for_Xs_detachment before the clip) and
// the ancestors-or-self of the start node (H0 / C0 are read off that path).
__device__ __forceinline__ bool branch_in_Xs_future(const ForestDev& f, const SprStudy& S, int p, int par) {
  if (par < 0 || p == S.posS || p == S.posP) return false;
  if (!(f.t[par] >= S.t_X)) return false;
  return !(p <= S.pos0 && S.pos0 < p + f.subtree_size[p]);
}

// Per-study view used by the scan / segments / emit kernels.  The tree prefix sums H_end, C_end and the kept-region base KB
// are stored two-level: a tile-local value per node plus one exclusive prefix per tile of kTile nodes (filled by
// spr_tile_prefix), so that no kernel ever waits on another CTA and nothing is rewritten in place.
struct SprView {
  const uint8_t* xtab;
  const int32_t* Hloc; const int32_t* Cloc; const int32_t* KBloc;
  const int32_t* agg;          // [num_tiles + 1][3]
  const int32_t* path; const int2* pae; const int32_t* seg;
  int node_base, path_len;
  int stride, shift;           // SprStudy::h_stride / tile_shift
  // event-scan grouped path: H and KB come from the group's event-prefix rows / keep masks (kernels_spr_group2.cuh)
  int g2, g2_lane, g2_mut_base, g2_num_templates;
  const int8_t* g2S; const int32_t* g2aggS; const uint32_t* g2mask; const int32_t* g2aggK;
  const int32_t* g2_eopen; const int32_t* g2_mut_off;
  // H_end(q): potential at the bottom of branch q == prefix of the signed events before event eopen(q) + np(q)
  __device__ __forceinline__ int H(int q) const {
    if (g2) {
      const int p = node_base + q;
      const int e = g2_eopen[p] + (g2_mut_off[p + 1] - g2_mut_off[p]);
      return (int)g2S[(size_t)e * 32 + g2_lane] + g2aggS[(size_t)(e >> 7) * 32 + g2_lane];
    }
    return Hloc[(size_t)q * stride] + agg[(q >> shift) * 3 + 0];
  }
  // H(q, k): potential of region k of branch q (event-scan path only): independent loads, no walk of the branch's mutations
  __device__ __forceinline__ int Hregion(int q, int k) const {
    const int e = g2_eopen[node_base + q] + k;
    return (int)g2S[(size_t)e * 32 + g2_lane] + g2aggS[(size_t)(e >> 7) * 32 + g2_lane];
  }
  __device__ __forceinline__ int C(int q) const { return Cloc[(size_t)q * stride] + agg[(q >> shift) * 3 + 1]; }
  // KB(q): kept regions of the positions before q (q == num_nodes allowed)
  __device__ __forceinline__ int KB(int q) const {
    if (g2) {
      const int p = node_base + q;
      const int tq = q + (g2_mut_off[p] - g2_mut_base);          // template index of region (q, 0); == num_templates for q == N
      const size_t w = (size_t)(tq >> 5) * 32 + g2_lane;
      return g2aggK[w] + __popc(g2mask[w] & ((1u << (tq & 31)) - 1u));
    }
    return KBloc[(size_t)q * stride] + agg[(q >> shift) * 3 + 2];
  }
};

__device__ __forceinline__ SprView make_view(const SprBatchDev& B, const SprStudy& S, int study) {
  SprView V;
  V.xtab = (const uint8_t*)(B.slab + S.off_xtab);
  V.Hloc = (const int32_t*)(B.slab + S.off_H);
  V.Cloc = (const int32_t*)(B.slab + S.off_C);
  V.KBloc = (const int32_t*)(B.slab + S.off_KB);
  V.agg = B.tile_agg + (size_t)study * (B.max_tiles + 1) * 3;
  V.path = (const int32_t*)(B.slab + S.off_path);
  V.pae = (const int2*)(B.slab + S.off_pae);
  V.seg = (const int32_t*)(B.slab + S.off_seg);
  V.node_base = S.node_base; V.path_len = S.path_len;
  V.stride = S.h_stride; V.shift = S.tile_shift;
  V.g2 = S.g2; V.g2_lane = S.g2_lane; V.g2_mut_base = S.g2_mut_base; V.g2_num_templates = S.g2_num_templates;
  V.g2S = (const int8_t*)(B.slab + S.off_g2S); V.g2aggS = (const int32_t*)(B.slab + S.off_g2aggS);
  V.g2mask = (const uint32_t*)(B.slab + S.off_g2mask); V.g2aggK = (const int32_t*)(B.slab + S.off_g2aggK);
  V.g2_eopen = B.g2_eopen; V.g2_mut_off = B.g2_mut_off;
  return V;
}

// deepest node of the start->root path that contains p in its subtree: binary search over the nested [start, end) ranges
__device__ __forceinline__ int classify(const SprView& V, int p) {
  int lo = 0, hi = V.path_len - 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const int2 ae = __ldg(V.pae + mid);
    if (p >= ae.x && p < ae.y) hi = mid; else lo = mid + 1;
  }
  return lo;
}

struct RegionEval { int branch, mut_idx; double t_min, t_max; bool keep; };

// Region (p,k) as the builder reports it AFTER account_for_Xs_detachment and remove_regions_in_Xs_future.
__device__ __forceinline__ RegionEval eval_region(const ForestDev& f, const SprStudy& S, int p, int k, int np, int moff,
                                                  double tPar, double tNode) {
  RegionEval r;
  r.branch = f.node_id[p];
  r.mut_idx = k;
  const bool is_root = (p == S.root_pos);
  r.t_min = is_root ? -DBL_MAX : (k == 0 ? tPar : f.mut_t[moff + k - 1]);       // spr_study.h:90-95
  r.t_max = is_root ? tNode : (k == np ? tNode : f.mut_t[moff + k]);            // spr_study.h:96-101
  r.keep = true;
  if (!S.can_change_root && is_root) r.keep = false;
  else if (S.posX >= 0 && (p == S.posS || p == S.posP)) {
    if (!S.P_is_root) {
      if (p == S.posS) {
        if (k == 0) {   // merged with the last region of P
          const int pm = f.mut_off[S.posP];
          r.t_min = S.nP == 0 ? f.t[f.parent_pos[S.posP]] : f.mut_t[pm + S.nP - 1];
        }
        r.mut_idx += S.nP;
      } else {
        if (k == S.nP) r.keep = false; else r.branch = f.node_id[S.posS];
      }
    } else if (S.can_change_root) {
      if (p == S.posS && k == S.nS) { r.mut_idx += S.nP; r.t_min = -DBL_MAX; }
      else r.keep = false;
    }
  }
  if (r.keep) {
    if (r.t_min >= S.t_X) r.keep = false;
    else if (r.t_max > S.t_X) r.t_max = S.t_X;
  }
  return r;
}

// counted-mutation distance from the start region; j = classify(p), Cd = C_down(p,k)
__device__ __forceinline__ int scope_dist(const SprView& V, int j, bool on_path, int Cd, int C0) {
  if (j == 0) return on_path ? abs(Cd - C0) : Cd - C0;
  if (on_path) return C0 - Cd;
  const int cj = V.C(V.path[j] - V.node_base);
  return (C0 - cj) + (Cd - cj);
}

// number of kept regions on branch p (all filters).  `limited` => needs the scope test.
__device__ int node_kept_count(const ForestDev& f, const SprStudy& S, const SprView& V, int p, bool limited, int C0) {
  if (S.posX >= 0 && p >= S.posX && p < S.posX + f.subtree_size[S.posX]) return 0;
  const int par = f.parent_pos[p];
  if (branch_in_Xs_future(f, S, p, par)) return 0;
  const int moff = f.mut_off[p], np = f.mut_off[p + 1] - moff;
  const double tNode = f.t[p], tPar = par >= 0 ? f.t[par] : 0.0;
  const bool is_root = p == S.root_pos;
  // an ordinary branch that ends before t_X keeps all of its np + 1 regions (t_min <= t_node < t_X)
  if (!limited && !is_root && p != S.posS && p != S.posP && tPar < S.t_X && tNode < S.t_X) return np + 1;
  int j = 0; bool on_path = false; int Cd = 0;
  if (limited) {
    j = classify(V, p);
    on_path = (V.path[j] == p);
    Cd = is_root ? 0 : V.C(par - S.node_base);
  }
  int cnt = 0;
  for (int k = is_root ? np : 0; k <= np; ++k) {
    bool ok = true;
    if (limited) {
      ok = scope_dist(V, j, on_path, Cd, C0) <= S.limit;
      if (k < np) { int dh, dc; mut_dc(V.xtab, f.mut_site[moff + k], f.mut_code[moff + k] & 15, dh, dc); Cd += dc; }
    }
    if (ok && eval_region(f, S, p, k, np, moff, tPar, tNode).keep) ++cnt;
  }
  return cnt;
}

// ---- (2) integer tree prefix sums H_end / C_end (+ kept-count scan when the study is unbounded) ------------------------------------
// H_end(q) = sum of the per-branch potentials dH over q and its ancestors.  In DFS pre-order that is the running sum of
// (dH of the node opening at q) - (dH of every node whose subtree closes right before q).  A node a closes right before position
// a + subtree_size[a], so each tile gathers its closers -- the contiguous slice post_node[c(first-1) .. c(last)) of the post-order
// list -- flat, one closer per thread, and subtracts them with shared-memory integer atomics (exact, order-free).  Closers that
// opened in an earlier tile recompute their potential from their own (short) mutation list.  No CTA waits on another one: each
// tile writes tile-local prefixes + its totals, and spr_tile_prefix turns the totals into per-tile exclusive prefixes.
// phase 0: H and C for every study; unbounded studies also get their kept-count scan here.
// phase 1: kept-count scan for bounded studies (needs the final C).
// A CTA of kTile threads covers kScanSub consecutive tiles (thread tid owns the kScanSub consecutive nodes tid * kScanSub ..,
// all inside one tile): the chain of dependent loads and the block-wide scans are paid once per 4 tiles, and the outputs keep
// their tile granularity (CTA-wide prefix minus the prefix at the tile's first node).
constexpr int kScanSub = 4;
constexpr int kScanNodes = kTile * kScanSub;

struct ScanSmem {
  SprStudy S;
  int h[kScanNodes], c[kScanNodes], dh[kScanNodes], dc[kScanNodes];
  int ws[kTile / 32];
  int bound[3][kScanSub + 1];      // CTA-wide inclusive prefix (H, C, kept) at the last node of each tile; [0] = 0
};

// CTA-wide inclusive scan of v[0..kScanSub) per thread (consecutive nodes); leaves the prefix at every tile end in bound[.]
__device__ __forceinline__ void cta_scan_tiles(int (&v)[kScanSub], int* ws, int* bound) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int mine = 0;
#pragma unroll
  for (int u = 0; u < kScanSub; ++u) mine += v[u];
  const int incl = warp_scan_incl(mine, lane);
  __syncthreads();                 // ws / bound may still be read from the previous scan
  if (lane == 31) ws[warp] = incl;
  __syncthreads();
  int run = incl - mine;
#pragma unroll
  for (int w = 0; w < kTile / 32; ++w) if (w < warp) run += ws[w];
#pragma unroll
  for (int u = 0; u < kScanSub; ++u) { run += v[u]; v[u] = run; }
  if (tid == 0) bound[0] = 0;
  if ((tid + 1) % (kTile / kScanSub) == 0) bound[(tid + 1) / (kTile / kScanSub)] = run;   // last node of a tile
  __syncthreads();
}

template <int kPhase>
__global__ void __launch_bounds__(kTile) spr_scan_kernel(ForestDev f, SprBatchDev B) {
  __shared__ ScanSmem sm;
  const int study = blockIdx.y;
  const int t0 = blockIdx.x * kScanSub;          // first tile of this CTA
  {
    const SprStudy& G = B.studies[study];
    if (t0 >= G.num_tiles || G.error || G.h_stride != 1) return;     // grouped studies are scanned by spr_g2_scan_kernel
    if (kPhase == 1 && G.limit == INT_MAX) return;
    const int* src = reinterpret_cast<const int*>(&G);
    int* dst = reinterpret_cast<int*>(&sm.S);
    for (int i = threadIdx.x; i < (int)(sizeof(SprStudy) / sizeof(int)); i += kTile) dst[i] = src[i];
  }
  __syncthreads();
  const SprStudy& S = sm.S;
  const bool limited = S.limit != INT_MAX;
  const int tid = threadIdx.x;
  const SprView V = make_view(B, S, study);
  int32_t* Hloc = (int32_t*)(B.slab + S.off_H);
  int32_t* Cloc = (int32_t*)(B.slab + S.off_C);
  int32_t* KBloc = (int32_t*)(B.slab + S.off_KB);
  int32_t* agg = B.tile_agg + ((size_t)study * (B.max_tiles + 1) + t0) * 3;
  const int node_base = S.node_base, N = S.num_nodes;
  const int cta_start = node_base + t0 * kTile;
  const int cta_end = min(cta_start + kScanNodes, node_base + N);
  const int n0 = tid * kScanSub;                 // my first node (CTA-local); all mine lie in tile `sub` of the CTA
  const int sub = n0 / kTile;
  const int ntiles = min(kScanSub, S.num_tiles - t0);

  if (kPhase == 0) {
    int par[kScanSub], kc[kScanSub];
    const int xs = S.posX, xe = S.posX >= 0 ? S.posX + f.subtree_size[S.posX] : -1;
#pragma unroll
    for (int u = 0; u < kScanSub; ++u) { const int p = cta_start + n0 + u; par[u] = p < cta_end ? f.parent_pos[p] : -1; }
#pragma unroll
    for (int u = 0; u < kScanSub; ++u) {
      const int p = cta_start + n0 + u;
      int dh = 0, dc = 0;
      kc[u] = 0;
      if (p < cta_end) {
        // one pass per node: the X's-future test (branch_in_Xs_future, inlined so that t[parent] is loaded once), the potentials of
        // its mutation list, and -- for unbounded studies -- its kept-region count
        const int pr = par[u];
        const bool is_root = pr < 0, special = p == S.posS || p == S.posP;
        const double tPar = is_root ? 0.0 : f.t[pr];
        const bool cut = !is_root && !special && tPar >= S.t_X && !(p <= S.pos0 && S.pos0 < p + f.subtree_size[p]);
        if (!cut) {
          const int moff = f.mut_off[p], np = f.mut_off[p + 1] - moff;
          if (!is_root) {          // the root's own list is never crossed by the walk
            for (int i = moff; i < moff + np; ++i) {
              int h, c;
              mut_dc(V.xtab, f.mut_site[i], f.mut_code[i] & 15, h, c);
              dh += h; dc += c;
            }
          }
          if (!limited && !(xs >= 0 && p >= xs && p < xe)) {
            // an ordinary branch that ends before t_X keeps all of its np + 1 regions (t_min <= t_node < t_X)
            if (!is_root && !special && tPar < S.t_X && f.t[p] < S.t_X) kc[u] = np + 1;
            else kc[u] = node_kept_count(f, S, V, p, false, 0);
          }
        }
      }
      sm.h[n0 + u] = dh; sm.c[n0 + u] = dc; sm.dh[n0 + u] = dh; sm.dc[n0 + u] = dc;
    }
    __syncthreads();
    {
      const int q_first = cta_start - node_base, q_last = cta_end - 1 - node_base;
      const int c0 = q_first == 0 ? 0 : (q_first - 1) - f.depth[cta_start - 1];
      const int c1 = q_last - f.depth[cta_end - 1];
      for (int j = c0 + tid; j < c1; j += kTile) {
        const int a = f.post_node[node_base + j];
        int ah, ac;
        if (a >= cta_start) { ah = sm.h[a - cta_start]; ac = sm.c[a - cta_start]; }
        else if (a == S.root_pos || branch_in_Xs_future(f, S, a, f.parent_pos[a])) { ah = 0; ac = 0; }
        else node_dc(f, V.xtab, a, ah, ac);
        const int qc = a + f.subtree_size[a] - cta_start;          // position right after a's subtree: inside this CTA's range
        if (ah) atomicSub(&sm.dh[qc], ah);
        if (limited && ac) atomicSub(&sm.dc[qc], ac);   // C (counted-mutation depth) only feeds the scope test of bounded studies
      }
    }
    __syncthreads();
    int vh[kScanSub], vc[kScanSub], vk[kScanSub];
#pragma unroll
    for (int u = 0; u < kScanSub; ++u) { vh[u] = sm.dh[n0 + u]; vc[u] = sm.dc[n0 + u]; vk[u] = kc[u]; }
    cta_scan_tiles(vh, sm.ws, sm.bound[0]);
    if (limited) cta_scan_tiles(vc, sm.ws, sm.bound[1]);
    if (!limited) cta_scan_tiles(vk, sm.ws, sm.bound[2]);
#pragma unroll
    for (int u = 0; u < kScanSub; ++u) {
      const int p = cta_start + n0 + u, q = p - node_base;
      if (p < cta_end) {
        Hloc[q] = vh[u] - sm.bound[0][sub];
        if (limited) Cloc[q] = vc[u] - sm.bound[1][sub];
        else {
          const int ik = vk[u] - sm.bound[2][sub];                  // tile-local inclusive
          KBloc[q] = ik - kc[u];
          if (q == N - 1) KBloc[N] = (N % kTile) ? ik : 0;          // KB(N): one past the end, same tile unless N is a tile multiple
        }
      }
    }
    if (tid < ntiles) {
      agg[tid * 3 + 0] = sm.bound[0][tid + 1] - sm.bound[0][tid];
      agg[tid * 3 + 1] = limited ? sm.bound[1][tid + 1] - sm.bound[1][tid] : 0;
      agg[tid * 3 + 2] = limited ? 0 : sm.bound[2][tid + 1] - sm.bound[2][tid];
    }
  } else {
    int vk[kScanSub], kc[kScanSub];
#pragma unroll
    for (int u = 0; u < kScanSub; ++u) { const int p = cta_start + n0 + u; kc[u] = p < cta_end ? node_kept_count(f, S, V, p, true, S.C0) : 0; vk[u] = kc[u]; }
    cta_scan_tiles(vk, sm.ws, sm.bound[2]);
#pragma unroll
    for (int u = 0; u < kScanSub; ++u) {
      const int p = cta_start + n0 + u, q = p - node_base;
      if (p < cta_end) {
        const int ik = vk[u] - sm.bound[2][sub];
        KBloc[q] = ik - kc[u];
        if (q == N - 1) KBloc[N] = (N % kTile) ? ik : 0;
      }
    }
    if (tid < ntiles) agg[tid * 3 + 2] = sm.bound[2][tid + 1] - sm.bound[2][tid];
  }
}

// Exclusive scan over the tiles of one study of the components in `want` that are not final yet (bit 0: H and C, bit 1: kept
// counts); entry [num_tiles] receives the totals.  Once H and C are final the start region's (C0, H0) are derived.  Called
// by a whole CTA of kSetupThreads threads; ends with a barrier.
__device__ void spr_tile_prefix(const ForestDev& f, SprBatchDev& B, SprStudy& S, int study, int want, int* s_ws, int* s_carry) {
  const int tid = threadIdx.x;
  const int todo = want & ~S.scanned;
  __syncthreads();
  if (todo == 0) return;
  int32_t* agg = B.tile_agg + (size_t)study * (B.max_tiles + 1) * 3;
  const int nt = S.num_htiles;
  for (int comp = 0; comp < 3; ++comp) {
    if (!((comp < 2 ? 1 : 2) & todo)) continue;
    if (tid == 0) *s_carry = 0;
    __syncthreads();
    for (int j0 = 0; j0 < nt; j0 += kSetupThreads) {
      const int j = j0 + tid;
      const int v = j < nt ? agg[j * 3 + comp] : 0;
      int tot;
      const int incl = block_scan_incl<int, kSetupThreads>(v, s_ws, &tot);
      if (j < nt) agg[j * 3 + comp] = *s_carry + incl - v;
      __syncthreads();
      if (tid == 0) *s_carry += tot;
      __syncthreads();
    }
    if (tid == 0) agg[nt * 3 + comp] = *s_carry;
    __syncthreads();
  }
  if (tid == 0) {
    if (todo & 1) {
      // C_down / H_down at the start region (pos0, k0)
      const SprView V = make_view(B, S, study);
      const int par = f.parent_pos[S.pos0];
      const bool top = par < 0 || S.pos0 == S.root_pos;
      int c = (top || S.limit == INT_MAX) ? 0 : V.C(par - S.node_base);
      int h = top ? 0 : V.H(par - S.node_base);
      if (S.pos0 != S.root_pos) {
        const int mo = f.mut_off[S.pos0];
        for (int i = 0; i < S.k0; ++i) { int dh, dc; mut_dc(V.xtab, f.mut_site[mo + i], f.mut_code[mo + i] & 15, dh, dc); c += dc; h += dh; }
      }
      S.C0 = c; S.H0 = h;
    }
    S.scanned |= todo;
    __threadfence_block();
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kSetupThreads) spr_tile_prefix_kernel(ForestDev f, SprBatchDev B) {
  __shared__ int s_ws[kSetupThreads / 32];
  __shared__ int s_carry;
  SprStudy& S = B.studies[blockIdx.x];
  if (S.error || S.h_stride == 0) return;              // (h_stride 0: the study is walked by spr_frontier_kernel)
  spr_tile_prefix(f, B, S, blockIdx.x, S.limit != INT_MAX ? 1 : 3, s_ws, &s_carry);
}

// ---- per-node emission under the general rules (grouped path: the root, P, S and the nodes of the start->root path) ------------------------
struct GLane {            // what a study carries through the grouped emit
  RegionHead* out;
  const int2* pae; const int32_t* seg;
  const int32_t* agg;
  int region_cap, path_len, H0, init_min_muts;
  double tX;
  double* lw; unsigned long long* max_key;      // fused weights: raw log-weights of the study, its running maximum (ordered key)
};

__device__ __forceinline__ void g_store_region(const GLane& L, int idx, int branch, int mut_idx, double t_min, double t_max, int m) {
  if (idx >= 0 && idx < L.region_cap) {
    // one 256-bit store per record (STG.256): in the grouped emit each lane writes into its own study's array, so every store
    // instruction of the warp touches 32 different lines -- halving the instructions halves the LSU wavefronts
    const unsigned long long w0 = (unsigned long long)(unsigned)branch | ((unsigned long long)(unsigned)mut_idx << 32);
    const unsigned long long w3 = (unsigned long long)(unsigned)m;
    asm volatile("st.global.v4.b64 [%0], {%1, %2, %3, %4};" ::"l"(L.out + idx), "l"(w0), "l"(__double_as_longlong(t_min)),
                 "l"(__double_as_longlong(t_max)), "l"(w3) : "memory");
  }
}

__device__ __noinline__ double region_log_W_above_root(double fa, double lam, double mu, double t_X, double t_max_tip, int m, double tS);

// Same arithmetic as the per-study emit kernel (eval_region + the segment bases), walking the node's regions in order.
// sg = the segment record of path index j = classify(p).  When the study's weights are fused into the emit (event-scan path), the
// raw log-weight of each of these few regions is written here as well (core/spr_study.cpp:306-376).
__device__ void g_emit_node_general(const ForestDev& f, const SprStudy& S, const SprView& V, const GLane& L, int p, const int32_t* sg, int j, bool on_path) {
  const int moff = f.mut_off[p], np = f.mut_off[p + 1] - moff;
  const int par = f.parent_pos[p];
  const bool is_root = p == S.root_pos;
  const double tNode = f.t[p], tPar = par >= 0 ? f.t[par] : 0.0;
  int Hk = (is_root || V.g2) ? 0 : V.H(par - S.node_base);
  const int kA = (j == 0) ? S.k0 : np;
  int n_up = 0, n_own = 0, rank = 0;
  unsigned long long best = 0ULL;       // fused weights: largest raw log-weight of this node's regions, as an ordered key
  const int base_off = on_path ? 0 : sg[2] - V.KB(sg[5] - S.node_base) + V.KB(p - S.node_base);
  for (int k = is_root ? np : 0; k <= np; ++k) {
    const RegionEval r = eval_region(f, S, p, k, np, moff, tPar, tNode);
    if (r.keep) {
      int idx;
      if (!on_path) idx = base_off + rank++;
      else if (k == kA) idx = sg[0];
      else if (k > kA) idx = sg[1] + n_own++;
      else idx = sg[3] + (sg[4] - 1 - n_up++);
      const int m = L.init_min_muts + ((V.g2 ? V.Hregion(p - S.node_base, k) : Hk) - L.H0);
      g_store_region(L, idx, r.branch, r.mut_idx, r.t_min, r.t_max, m);
      if (S.weights_fused && idx >= 0 && idx < L.region_cap) {
        double lw;
        if (r.t_min != -DBL_MAX) {
          const double t_prime = 0.5 * (r.t_min + r.t_max);
          lw = log(S.f * S.lambda_X * (r.t_max - r.t_min)) + S.f * (-S.lambda_X * (S.t_X - t_prime) + m * log(S.mu * (S.t_X - t_prime) / 3));
        } else {
          lw = region_log_W_above_root(S.f, S.lambda_X, S.mu, S.t_X, S.t_max_tip, m, f.t[S.node_base + f.pos_of_node[S.node_base + r.branch]]);
        }
        L.lw[idx] = lw;
        if (lw == lw) { const unsigned long long key = f64_order_key(lw); if (key > best) best = key; }
      }
    }
    if (!V.g2 && k < np && !is_root) { int dh, dc; mut_dc(V.xtab, f.mut_site[moff + k], f.mut_code[moff + k] & 15, dh, dc); Hk += dh; }
  }
  if (best != 0ULL) atomicMax(L.max_key, best);
}

// ---- (3) segment bases along the start->root path ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kSetupThreads) spr_segments_kernel(ForestDev f, SprBatchDev B) {
  __shared__ int s_ws[kSetupThreads / 32];
  __shared__ int s_carry;
  // the study record, read once: every region evaluated below consults a dozen of its fields, and a reference into global memory
  // would re-load each of them after every store
  __shared__ SprStudy sS;
  SprStudy& Sg = B.studies[blockIdx.x];
  if (Sg.error || Sg.h_stride == 0) return;            // (h_stride 0: the study is walked by spr_frontier_kernel)
  static_assert(sizeof(SprStudy) % sizeof(int) == 0, "SprStudy is copied word by word");
  for (int i = threadIdx.x; i < (int)(sizeof(SprStudy) / sizeof(int)); i += kSetupThreads) reinterpret_cast<int*>(&sS)[i] = reinterpret_cast<const int*>(&Sg)[i];
  __syncthreads();
  const SprStudy& S = sS;
  if (threadIdx.x == 0) { const double mu = S.lambda_X / (double)(S.L - S.num_missing); sS.mu = mu; Sg.mu = mu; }   // Spr_study::mu, core/spr_study.cpp:239
  // the path index of S and P (a ten-step search of dependent loads) is found now, by two threads of another warp, rather than at the
  // end of the kernel where it would sit on the critical path
  __shared__ int s_jsp[2];
  if (S.h_stride != 1 && (threadIdx.x == 32 || threadIdx.x == 33)) {
    const int p = threadIdx.x == 32 ? S.posS : S.posP;
    s_jsp[threadIdx.x - 32] = p >= 0 ? classify(make_view(B, S, blockIdx.x), p) : 0;
  }
  if (S.g2) {
    // event-scan path: the chunk prefixes are already final (spr_g2_prefix_kernel); only the start region's potential is missing
    if (threadIdx.x == 0) {
      const SprView V0 = make_view(B, S, blockIdx.x);
      const int par = f.parent_pos[S.pos0];
      const bool top = par < 0 || S.pos0 == S.root_pos;
      int h = top ? 0 : V0.H(par - S.node_base);
      if (S.pos0 != S.root_pos) {
        const int mo = f.mut_off[S.pos0];
        for (int i = 0; i < S.k0; ++i) { int dh, dc; mut_dc(V0.xtab, f.mut_site[mo + i], f.mut_code[mo + i] & 15, dh, dc); h += dh; }
      }
      Sg.C0 = 0; Sg.H0 = h; Sg.scanned = 3;
      sS.C0 = 0; sS.H0 = h; sS.scanned = 3;
      __threadfence_block();
    }
    __syncthreads();
  } else {
    spr_tile_prefix(f, B, Sg, blockIdx.x, 3, s_ws, &s_carry);
    if (threadIdx.x == 0) { sS.C0 = Sg.C0; sS.H0 = Sg.H0; sS.scanned = Sg.scanned; }
    __syncthreads();
  }
  const int tid = threadIdx.x;
  const SprView V = make_view(B, S, blockIdx.x);
  int32_t* seg = (int32_t*)(B.slab + S.off_seg);
  const bool limited = S.limit != INT_MAX;
  const int C0 = S.C0;
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (int j0 = 0; j0 < S.path_len; j0 += kSetupThreads) {
    const int j = j0 + tid;
    int cntA = 0, cntOwn = 0, cntSub = 0, cntUp = 0, sibpos = -1;
    if (j < S.path_len) {
      const int a = V.path[j];
      const int moff = f.mut_off[a], np = f.mut_off[a + 1] - moff;
      const int par = f.parent_pos[a];
      const bool is_root = a == S.root_pos;
      const double tNode = f.t[a], tPar = par >= 0 ? f.t[par] : 0.0;
      int Cd = (is_root || !limited) ? 0 : V.C(par - S.node_base);
      const int kA = (j == 0) ? S.k0 : np;
      for (int k = is_root ? np : 0; k <= np; ++k) {
        bool ok = true;
        if (limited) {
          ok = scope_dist(V, j, true, Cd, C0) <= S.limit;
          if (k < np) { int dh, dc; mut_dc(V.xtab, f.mut_site[moff + k], f.mut_code[moff + k] & 15, dh, dc); Cd += dc; }
        }
        if (ok && eval_region(f, S, a, k, np, moff, tPar, tNode).keep) {
          if (k == kA) ++cntA; else if (k < kA) ++cntUp; else ++cntOwn;
        }
      }
      const int qa = a - S.node_base;
      if (j == 0) {
        sibpos = a + 1;
        cntSub = V.KB(qa + f.subtree_size[a]) - V.KB(qa + 1);
      } else {
        const int c1 = a + 1, c0 = a + 1 + f.subtree_size[a + 1];
        sibpos = (V.path[j - 1] == c1) ? c0 : c1;
        const int qs = sibpos - S.node_base;
        cntSub = V.KB(qs + f.subtree_size[sibpos]) - V.KB(qs);
      }
    }
    const int tot = cntA + cntOwn + cntSub + cntUp;
    int btot;
    const int incl = block_scan_incl<int, kSetupThreads>(tot, s_ws, &btot);
    const int base = s_carry + incl - tot;
    if (j < S.path_len) {
      int32_t* sg = seg + (size_t)j * kSegStride;
      sg[0] = base; sg[1] = base + cntA; sg[2] = base + cntA + cntOwn; sg[3] = base + cntA + cntOwn + cntSub;
      sg[4] = cntUp; sg[5] = sibpos;
      // output offset of the regions hanging off path node j, relative to the kept-region prefix KB (spr_g2_bases_kernel / emit)
      if (S.g2) ((int32_t*)(B.slab + S.off_hang))[j] = sg[2] - V.KB(sibpos - S.node_base);
      if (S.h_stride != 1) {
        // grouped studies: the path nodes' own regions are written here, one thread per path node (spr_g2_emit_kernel skips them)
        GLane L;
        L.out = (RegionHead*)(B.slab + S.off_regions); L.pae = V.pae; L.seg = V.seg; L.agg = V.agg;
        L.region_cap = S.region_cap; L.path_len = S.path_len; L.H0 = S.H0; L.init_min_muts = S.init_min_muts; L.tX = S.t_X;
        L.lw = (double*)(B.slab + S.off_lw); L.max_key = &Sg.max_key;
        g_emit_node_general(f, S, V, L, V.path[j], sg, j, true);
      }
    }
    __syncthreads();
    if (tid == 0) s_carry += btot;
    __syncthreads();
  }
  if (tid == 0) Sg.total_regions = s_carry;
  if (S.h_stride != 1 && tid < 2) {
    // ... and so are S and P when they are not on the path (their regions are relabelled by account_for_Xs_detachment)
    const int p = tid == 0 ? S.posS : S.posP;
    if (p >= 0 && !(tid == 1 && S.posP == S.posS)) {
      const int j = s_jsp[tid];
      if (V.path[j] != p) {
        GLane L;
        L.out = (RegionHead*)(B.slab + S.off_regions); L.pae = V.pae; L.seg = V.seg; L.agg = V.agg;
        L.region_cap = S.region_cap; L.path_len = S.path_len; L.H0 = S.H0; L.init_min_muts = S.init_min_muts; L.tX = S.t_X;
        L.lw = (double*)(B.slab + S.off_lw); L.max_key = &Sg.max_key;
        g_emit_node_general(f, S, V, L, p, seg + (size_t)j * kSegStride, j, false);
      }
    }
  }
  // classify() of the first and the last node of every tile: the deepest path node containing p is monotone in p on either side
  // of the start node, so these bracket the search of every node of the tile (spr_emit_kernel)
  int2* tj = (int2*)(B.slab + S.off_tj);
  if (S.h_stride == 1)
  for (int t = tid; t < S.num_tiles; t += kSetupThreads) {
    const int first = S.node_base + t * kTile, last = min(first + kTile, S.node_base + S.num_nodes) - 1;
    tj[t] = make_int2(classify(V, first), classify(V, last));
  }
}

// ---- fp64 log for the region weights -----------------------------------------------------------------------------------------------------
// Two logs per candidate region are most of the arithmetic of the weight pass (the library routine is ~100 instructions).  The
// weights are compared at 1e-9 relative (BASELINE.json north_star), so a 128-entry table of (1/c, log c) over the mantissa's top
// 7 bits + a degree-6 polynomial of r = m/c - 1 (|r| <= 2^-8, truncation 2^-56) + a two-part ln 2 is ample: absolute error
// < 5e-16 on [1e-12, 1e3], ~1e-15 relative to a weight exponent of O(10).  Zero, denormal, infinite, NaN and negative arguments go to
// the library routine, so -inf for an empty region is preserved (core/spr_study.cpp:318).
constexpr int kLogTabBits = 7;
__device__ __forceinline__ void fill_log_table(double2* tab) {
  for (int i = threadIdx.x; i < (1 << kLogTabBits); i += blockDim.x) {
    const double c = 1.0 + (i + 0.5) / (double)(1 << kLogTabBits);
    tab[i] = make_double2(1.0 / c, log(c));
  }
}
__device__ __forceinline__ double fast_log(double x, const double2* __restrict__ tab) {
  const long long b = __double_as_longlong(x);
  const int hi = (int)(b >> 32);
  const int ex = (hi >> 20) & 0x7ff;
  if (ex == 0 || ex == 0x7ff || hi < 0) return log(x);
  const double2 tc = tab[(hi >> (20 - kLogTabBits)) & ((1 << kLogTabBits) - 1)];
  const double m = __longlong_as_double((b & 0x000fffffffffffffLL) | 0x3ff0000000000000LL);
  const double r = fma(m, tc.x, -1.0);
  double p = fma(r, -1.0 / 6.0, 0.2);
  p = fma(r, p, -0.25); p = fma(r, p, 1.0 / 3.0); p = fma(r, p, -0.5); p = fma(r, p, 1.0);
  const double e = (double)(ex - 1023);
  return fma(e, 6.93147180369123816490e-01, fma(e, 1.90821492927058770002e-10, fma(r, p, tc.y)));
}

// ---- (4) emit regions in the reference's DFS order, with raw log-weights ------------------------------------------------------------------
// above-root region (core/spr_study.cpp:334-369): one region per study at most, kept out of line so that its lgamma /
// incomplete-gamma code does not inflate the register budget of the common path
__device__ __noinline__ double region_log_W_above_root(double fa, double lam, double mu, double t_X, double t_max_tip, int m, double tS) {
  const double s_min = fabs(t_X - tS);
  const double t_early = fmin(t_X, tS);
  const double s_max = s_min + 20.0 * (t_max_tip - t_early);
  const double x_min = lam * fa * s_min, x_max = lam * fa * s_max;
  if (x_max < 0.01) {
    const double alpha = fa * m + 1;
    return -0.6931471805599453 + log(fa * lam) + fa * m * log(mu / 3) + alpha * log(s_max) + log1p(-pow(s_min / s_max, alpha)) - log(alpha);
  }
  const double a = fa * m + 1;
  return -0.6931471805599453 + fa * m * log(mu / (3 * lam * fa)) + lgamma(a) + log(dev_gamma_q(a, x_min) - dev_gamma_q(a, x_max));
}

// Two phases per tile of kTile nodes.  (A) one thread per node: the node's record (list range, H / C at its parent, times,
// segment constants) goes to shared memory and the per-node candidate counts (np + 1 regions; 1 for the root) are scanned into
// slot offsets; the tile's mutations -- one contiguous CSR range -- get their (dH, counted) pair flat, one per thread.
// (B) one thread per SLOT (= candidate region), in rounds of kTile: the slot finds its node by binary search in the slot
// offsets, so the expensive part of a region (keep rules, two fp64 logs, three 16-byte stores) runs with all lanes busy
// no matter how the mutations are distributed over the nodes.  For regions off the start->root path the output index is
//   seg[2] - KB(sibling) + (KB(tile) + rank of the kept region inside the tile)
// i.e. one ballot-scan of the keep flags per round; consecutive kept slots write consecutive 48-byte records.
constexpr int kEmitSub = 4;                    // kTile-tiles per CTA: the per-CTA chain of dependent loads is amortised over 4x the nodes
constexpr int kEmitNodes = kTile * kEmitSub;
constexpr int kEmitMutCap = 4096;              // per-CTA mutations whose (dH, counted) pair is cached in shared memory

struct EmitSmem {
  SprStudy S;                                  // the study record, read once (it lives in global memory)
  int start[kEmitNodes + 1];                   // exclusive scan of the per-node candidate counts
  int moff[kEmitNodes], np[kEmitNodes], Hpar[kEmitNodes], Cpar[kEmitNodes], hang[kEmitNodes], cls[kEmitNodes];   // cls = j << 1 | on_path
  int wcnt[kTile / 32];
  signed char dhc[kEmitMutCap];                // (dH + 1) | counted << 2
};

__device__ __forceinline__ void emit_mut_dc(const ForestDev& f, const EmitSmem& sm, const uint8_t* __restrict__ xtab, int m0, int i, int& dh, int& dc) {
  const int rel = i - m0;
  if (rel < kEmitMutCap) { const int v = sm.dhc[rel]; dh = (v & 3) - 1; dc = v >> 2; }
  else mut_dc(xtab, f.mut_site[i], f.mut_code[i] & 15, dh, dc);
}

// 4 resident CTAs per SM: 64 registers, 16 bytes of spill stores (5 or 6 CTAs: 48 / 40 registers, 36 / 192 bytes)
__global__ void __launch_bounds__(kTile, 4) spr_emit_kernel(ForestDev f, SprBatchDev B) {
  __shared__ EmitSmem sm;
  const int study = blockIdx.y;
  const int t0 = blockIdx.x * kEmitSub;        // first kTile-tile of this CTA
  {
    const SprStudy& G = B.studies[study];
    if (t0 >= G.num_tiles || G.error || G.h_stride != 1) return;     // grouped studies are emitted by spr_g2_emit_kernel
    const int* src = reinterpret_cast<const int*>(&G);
    int* dst = reinterpret_cast<int*>(&sm.S);
    for (int i = threadIdx.x; i < (int)(sizeof(SprStudy) / sizeof(int)); i += kTile) dst[i] = src[i];
  }
  __syncthreads();
  const SprStudy& S = sm.S;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const SprView V = make_view(B, S, study);
  RegionHead* out = (RegionHead*)(B.slab + S.off_regions);
  const bool limited = S.limit != INT_MAX;
  const int C0 = S.C0, H0 = S.H0;
  const int t1 = min(t0 + kEmitSub, S.num_tiles);
  const int kb_first = V.agg[t0 * 3 + 2];       // kept regions before this CTA's nodes (KBloc of a tile's first node is 0)
  if (V.agg[t1 * 3 + 2] == kb_first) return;    // nothing kept here (X's subtree, X's future, out of scope)
  const int cta_start = S.node_base + t0 * kTile;
  const int cta_end = min(cta_start + kEmitNodes, S.node_base + S.num_nodes);
  const int xs = S.posX, xe = S.posX >= 0 ? S.posX + f.subtree_size[S.posX] : -1;
  const int2* tj = (const int2*)(B.slab + S.off_tj);
  const int jb0 = __ldg(&tj[t0].x), jb1 = __ldg(&tj[t1 - 1].y);
  const int m0 = f.mut_off[cta_start], m1 = f.mut_off[cta_end];
  for (int g = m0 + tid; g < min(m1, m0 + kEmitMutCap); g += kTile) {
    int dh, dc; mut_dc(V.xtab, f.mut_site[g], f.mut_code[g] & 15, dh, dc);
    sm.dhc[g - m0] = (signed char)((dh + 1) | (dc << 2));
  }

  // ---- (A) node records + slot offsets: thread tid owns the kEmitSub consecutive nodes tid * kEmitSub .. ------------------------------
  int cnt[kEmitSub];
  int par[kEmitSub];
#pragma unroll
  for (int u = 0; u < kEmitSub; ++u) { const int p = cta_start + tid * kEmitSub + u; par[u] = p < cta_end ? f.parent_pos[p] : -1; }
#pragma unroll
  for (int u = 0; u < kEmitSub; ++u) {
    const int n = tid * kEmitSub + u, p = cta_start + n;
    cnt[u] = 0;
    if (p < cta_end && !(xs >= 0 && p >= xs && p < xe) && !branch_in_Xs_future(f, S, p, par[u])) {
      const int moff = f.mut_off[p], np = f.mut_off[p + 1] - moff;
      const bool is_root = p == S.root_pos;
      int lo = min(jb0, jb1), hi = max(jb0, jb1);
      if (cta_start <= S.pos0 && S.pos0 < cta_end) lo = 0;       // the CTA holds the start node: both sides of the bracket
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const int2 ae = __ldg(V.pae + mid);
        if (p >= ae.x && p < ae.y) hi = mid; else lo = mid + 1;
      }
      const int j = lo;
      const bool on_path = V.path[j] == p;
      const int32_t* sg = V.seg + (size_t)j * kSegStride;
      sm.moff[n] = moff; sm.np[n] = np;
      sm.Hpar[n] = is_root ? 0 : V.H(par[u] - S.node_base);
      sm.Cpar[n] = (limited && !is_root) ? V.C(par[u] - S.node_base) : 0;
      sm.hang[n] = on_path ? 0 : sg[2] - V.KB(sg[5] - S.node_base);
      sm.cls[n] = (j << 1) | (on_path ? 1 : 0);
      cnt[u] = is_root ? 1 : np + 1;
    }
  }
  {
    int mine = 0;
#pragma unroll
    for (int u = 0; u < kEmitSub; ++u) mine += cnt[u];
    const int incl = warp_scan_incl(mine, lane);
    if (lane == 31) sm.wcnt[warp] = incl;
    __syncthreads();
    int run = incl - mine;
#pragma unroll
    for (int w = 0; w < kTile / 32; ++w) if (w < warp) run += sm.wcnt[w];
#pragma unroll
    for (int u = 0; u < kEmitSub; ++u) { sm.start[tid * kEmitSub + u] = run; run += cnt[u]; }
    if (tid == kTile - 1) sm.start[kEmitNodes] = run;
    __syncthreads();
  }
  const int total = sm.start[kEmitNodes];

  // ---- (B) one slot per thread ------------------------------------------------------------------------------------------------------------
  int carry = 0;
  for (int s0 = 0; s0 < total; s0 += kTile) {
    const int s = s0 + tid;
    bool keep = false;
    int n = 0, k = 0, Hk = 0, j = 0;
    bool on_path = false;
    double tNode = 0.0, tPar = 0.0;
    RegionEval r{};
    if (s < total) {
      int lo = 0, hi = kEmitNodes - 1;                // last node with start <= s (nodes with no slot share their successor's start)
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (sm.start[mid] <= s) lo = mid; else hi = mid - 1;
      }
      n = lo;
      const int pn = cta_start + n;
      const int np = sm.np[n], moff = sm.moff[n];
      const bool is_root = pn == S.root_pos;
      k = is_root ? np : s - sm.start[n];
      Hk = sm.Hpar[n];
      int Ck = sm.Cpar[n];
      const int ncross = is_root ? 0 : k;             // the root's own list is never crossed by the walk
      for (int i = 0; i < ncross; ++i) { int dh, dc; emit_mut_dc(f, sm, V.xtab, m0, moff + i, dh, dc); Hk += dh; Ck += dc; }
      j = sm.cls[n] >> 1; on_path = sm.cls[n] & 1;
      bool ok = true;
      if (limited) ok = scope_dist(V, j, on_path, Ck, C0) <= S.limit;
      if (ok) {
        const int pp = f.parent_pos[pn];
        tNode = f.t[pn]; tPar = pp >= 0 ? f.t[pp] : 0.0;
        r = eval_region(f, S, pn, k, np, moff, tPar, tNode); keep = r.keep;
      }
    }
    // rank of the kept slot inside the CTA's node range (ballot scan)
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) sm.wcnt[warp] = __popc(bal);
    __syncthreads();
    int pre = 0, rtot = 0;
#pragma unroll
    for (int w = 0; w < kTile / 32; ++w) { const int c = sm.wcnt[w]; if (w < warp) pre += c; rtot += c; }
    const int rank = carry + pre + __popc(bal & ((1u << lane) - 1u));
    carry += rtot;
    __syncthreads();                                  // wcnt is rewritten by the next round
    if (keep) {
      int idx;
      if (!on_path) idx = sm.hang[n] + kb_first + rank;
      else {
        // a node of the start->root path (at most depth-many per study): its regions go to the path segments
        const int pn = cta_start + n, np = sm.np[n], moff = sm.moff[n];
        const int32_t* sg = V.seg + (size_t)j * kSegStride;
        const int kA = (j == 0) ? S.k0 : np;
        if (k == kA) idx = sg[0];
        else {
          int before = 0, Ck = sm.Cpar[n];
          const int kfirst = (pn == S.root_pos) ? np : 0;
          for (int k2 = kfirst; k2 < k; ++k2) {
            bool ok2 = true;
            if (limited) ok2 = scope_dist(V, j, true, Ck, C0) <= S.limit;
            if (k2 < np) { int dh, dc; emit_mut_dc(f, sm, V.xtab, m0, moff + k2, dh, dc); Ck += dc; }
            if (ok2 && (k > kA ? k2 > kA : true) && eval_region(f, S, pn, k2, np, moff, tPar, tNode).keep) ++before;
          }
          idx = k > kA ? sg[1] + before : sg[3] + (sg[4] - 1 - before);
        }
      }
      const int m = S.init_min_muts + (Hk - H0);
      if (idx >= 0 && idx < S.region_cap) {
        // the 32-byte head as two 16-byte stores (one whole sector); the weights are a separate streaming pass over the heads
        // (spr_weights_kernel), as they are a separate step in the reference (the Spr_study constructor, core/spr_study.cpp:226-385)
        int4* o = reinterpret_cast<int4*>(out + idx);
        o[0] = make_int4(r.branch, r.mut_idx, __double2loint(r.t_min), __double2hiint(r.t_min));
        o[1] = make_int4(__double2loint(r.t_max), __double2hiint(r.t_max), m, 0);
      }
    }
  }
}

// ---- (4b) raw log-weights of the emitted regions + their maximum (Spr_study::Spr_study, core/spr_study.cpp:306-376) ----------------------
// Flat over regions: each thread reads one 32-byte head, writes one 8-byte raw log-weight; block maximum -> one ordered-integer
// atomicMax per CTA (exact, order independent).  The above-root region needs t_S = t[region.branch]: one gather per study at most.
constexpr int kWeightBlocks = 128;
__device__ __forceinline__ void ld_head_256(const RegionHead* p, unsigned long long& w0, double& t_min, double& t_max, unsigned long long& w3) {
  long long a, b;
  asm volatile("ld.global.nc.L1::no_allocate.v4.b64 {%0, %1, %2, %3}, [%4];" : "=l"(w0), "=l"(a), "=l"(b), "=l"(w3) : "l"(p));
  t_min = __longlong_as_double(a); t_max = __longlong_as_double(b);
}
__global__ void __launch_bounds__(256, 4) spr_weights_kernel(ForestDev f, SprBatchDev B) {
  __shared__ double s_ws[8];
  __shared__ double2 s_log[1 << kLogTabBits];
  fill_log_table(s_log);
  __syncthreads();
  const int study = blockIdx.y;
  const SprStudy& S = B.studies[study];
  if (S.error || !(S.lambda_X > 0.0) || S.weights_fused) return;
  const int n = min(S.total_regions, S.region_cap);
  const RegionHead* __restrict__ heads = (const RegionHead*)(B.slab + S.off_regions);
  double* __restrict__ lw_out = (double*)(B.slab + S.off_lw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // the study's constants in registers: the stores below could alias the study record as far as the compiler knows
  const double fa = S.f, lam = S.lambda_X, tX = S.t_X, mu = S.mu, falam = fa * lam;
  double wmax = -CUDART_INF;
  bool any = false;
  int root_i = -1, root_m = 0, root_branch = 0;      // the above-root region (one per study at most) is finished after the loop
  auto one = [&](int i, unsigned long long w0, double t_min, double t_max, unsigned long long w3) {
    const int m = (int)(unsigned)w3;
    if (t_min != -DBL_MAX) {
      // core/spr_study.cpp:313-318
      const double t_prime = 0.5 * (t_min + t_max);
      const double lw = fast_log(falam * (t_max - t_min), s_log) + fa * (-lam * (tX - t_prime) + m * fast_log(mu * (tX - t_prime) / 3, s_log));
      lw_out[i] = lw;
      wmax = any ? fmax(wmax, lw) : lw;   // std::max semantics of the reference's running maximum
      any = true;
    } else {
      root_i = i; root_m = m; root_branch = (int)(unsigned)w0;
    }
  };
  // two regions per thread per round: both 32-byte heads are in flight before the first logarithm starts
  int i = blockIdx.x * 256 + threadIdx.x;
  for (; i + kWeightBlocks * 256 < n; i += 2 * kWeightBlocks * 256) {
    unsigned long long a0, a3, b0, b3; double a1, a2, b1, b2;
    ld_head_256(heads + i, a0, a1, a2, a3);
    ld_head_256(heads + i + kWeightBlocks * 256, b0, b1, b2, b3);
    one(i, a0, a1, a2, a3);
    one(i + kWeightBlocks * 256, b0, b1, b2, b3);
  }
  if (i < n) {
    unsigned long long a0, a3; double a1, a2;
    ld_head_256(heads + i, a0, a1, a2, a3);
    one(i, a0, a1, a2, a3);
  }
  if (root_i >= 0) {
    const double lw = region_log_W_above_root(fa, lam, mu, tX, S.t_max_tip, root_m, f.t[S.node_base + f.pos_of_node[S.node_base + root_branch]]);
    lw_out[root_i] = lw;
    wmax = any ? fmax(wmax, lw) : lw;
  }
  double wm = warp_max(wmax);
  if (lane == 0) s_ws[warp] = wm;
  __syncthreads();
  if (warp == 0) {
    wm = lane < 8 ? s_ws[lane] : -CUDART_INF;
    wm = warp_max(wm);
    if (lane == 0 && wm > -CUDART_INF) atomicMax(&B.studies[study].max_key, f64_order_key(wm));
  }
}

// new (lambda_X, f, t_max_tip) for studies whose regions are already enumerated: dphy_spr_batch_set_weights
__global__ void spr_set_weight_params_kernel(ForestDev f, SprBatchDev B, const double* __restrict__ wp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B.num_studies) return;
  SprStudy& S = B.studies[i];
  S.lambda_X = wp[3 * i]; S.f = wp[3 * i + 1]; S.t_max_tip = wp[3 * i + 2];
  S.mu = S.lambda_X / (double)(S.L - S.num_missing);
  S.max_key = 0ULL; S.log_Wmax = 0.0; S.sum_W = 0.0;
  S.weights_fused = 0;      // the weights pass over the stored heads does it this time
}

// ---- (5) normalise: log_W_over_Wmax -= log_Wmax; W = exp(.); sum in a fixed order ------------------------------------------------------------
__global__ void __launch_bounds__(256) spr_normalize_kernel(SprBatchDev B) {
  __shared__ double s_ws[8];
  __shared__ int s_last;
  const int study = blockIdx.y;
  SprStudy& S = B.studies[study];
  if (S.error || !(S.lambda_X > 0.0)) return;
  const int n = min(S.total_regions, S.region_cap);
  double2* __restrict__ nw = (double2*)(B.slab + S.off_nw);
  double* part = (double*)(B.slab + S.off_part);
  const double lmax = n > 0 ? f64_from_order_key(S.max_key) : 0.0;
  const int per = (((n + kNormBlocks - 1) / kNormBlocks) + 1) & ~1;      // even: every block starts on a 16-byte boundary of lw_raw
  const int i0 = min((int)blockIdx.x * per, n), i1 = min(i0 + per, n);
  double acc = 0.0;
  const double* __restrict__ lw_raw = (const double*)(B.slab + S.off_lw);
  // a pair of regions per thread and four pairs in flight per round: 16-byte loads, 32-byte (whole-sector) stores; the summation
  // order is fixed by (n, grid), so sum_W is bit-reproducible
  constexpr int kU = 4;
  for (int b0 = i0; b0 < i1; b0 += 2 * 256 * kU) {
    double2 v[kU];
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      const int i = b0 + 2 * (u * 256 + (int)threadIdx.x);
      v[u] = make_double2(0.0, 0.0);
      if (i + 1 < i1) v[u] = __ldcs(reinterpret_cast<const double2*>(lw_raw + i));
      else if (i < i1) v[u].x = __ldcs(lw_raw + i);
    }
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      const int i = b0 + 2 * (u * 256 + (int)threadIdx.x);
      if (i < i1) {
        const double la = v[u].x - lmax, wa = exp(la);
        acc += wa;
        if (i + 1 < i1) {
          const double lb = v[u].y - lmax, wb = exp(lb);
          acc += wb;
          // (log_W_over_Wmax, W_over_Wmax) of two consecutive regions: one 32-byte store
          asm volatile("st.global.cs.v4.b64 [%0], {%1, %2, %3, %4};" ::"l"(nw + i), "l"(__double_as_longlong(la)), "l"(__double_as_longlong(wa)),
                       "l"(__double_as_longlong(lb)), "l"(__double_as_longlong(wb)) : "memory");
        } else {
          nw[i] = make_double2(la, wa);
        }
      }
    }
  }
  acc = block_sum<double, 256>(acc, s_ws);
  if (threadIdx.x == 0) {
    part[blockIdx.x] = acc;
    __threadfence();
    const uint32_t done = atomicAdd(B.ticket + study * 4 + 2, 1u);
    s_last = done == kNormBlocks - 1;
  }
  __syncthreads();
  if (s_last && threadIdx.x == 0) {
    __threadfence();
    double s = 0.0;
    for (int b = 0; b < kNormBlocks; ++b) s += ld_cg_f64(part + b);
    S.sum_W = s;
    S.log_Wmax = lmax;
    B.ticket[study * 4 + 2] = 0u;
  }
}

#include "kernels_spr_group.cuh"
#include "kernels_spr_group2.cuh"
#include "kernels_spr_frontier.cuh"

// ---- pick_nexus_region / find_region ------------------------------------------------------------------------------------------------------------------
// Spr_study::pick_nexus_region (core/spr_study.cpp:404-422) scans "if (W_i >= r) pick i; else r -= W_i": a chain of fp64 subtractions
// whose rounding decides the index when r falls next to a boundary.  A prefix sum in any other association can pick the neighbour
// (round 1 did, and its test allowed it), so the scan is replayed in the reference's own order: one warp per study, the weights
// loaded 32 at a time (the next chunk already in flight), every lane carrying the same r.  ~1 ms for the studies of a batch, once
// per study at most.
__global__ void __launch_bounds__(128) spr_pick_kernel(SprBatchDev B, const double* __restrict__ r_in, int32_t* __restrict__ out_idx) {
  const unsigned full = 0xffffffffu;
  const int study = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (study >= B.num_studies) return;
  const SprStudy& S = B.studies[study];
  const int n = min(S.total_regions, S.region_cap);
  const double2* __restrict__ nw = (const double2*)(B.slab + S.off_nw);
  double r = r_in[study];
  int found = -1;
  double w_next = lane < n ? nw[lane].y : 0.0;
  for (int i0 = 0; i0 < n && found < 0; i0 += 32) {
    const double w = w_next;
    w_next = i0 + 32 + lane < n ? nw[i0 + 32 + lane].y : 0.0;
    const int cnt = min(32, n - i0);
    for (int j = 0; j < cnt; ++j) {
      const double wj = __shfl_sync(full, w, j);
      if (wj >= r) { found = i0 + j; break; }
      r -= wj;
    }
  }
  if (lane == 0) out_idx[study] = found < 0 ? 0 : found;
}

__global__ void __launch_bounds__(256) spr_find_kernel(SprBatchDev B, int study, int branch, double t, int32_t* out_idx) {
  const SprStudy& S = B.studies[study];
  const int n = min(S.total_regions, S.region_cap);
  const RegionHead* reg = (const RegionHead*)(B.slab + S.off_regions);
  for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256)
    if (reg[i].branch == branch && reg[i].t_min < t && t <= reg[i].t_max) atomicMin(out_idx, i);
}

// ---- Spr_study::log_alpha_in_region (core/spr_study.cpp:486-549): one region, one thread ------------------------------------------------------
__global__ void spr_log_alpha_kernel(ForestDev f, SprBatchDev B, int study, int idx, double t, double* out) {
  const SprStudy& S = B.studies[study];
  const RegionHead rg = ((const RegionHead*)(B.slab + S.off_regions))[idx];
  const double2 nw = ((const double2*)(B.slab + S.off_nw))[idx];
  const double log_p_region = nw.x - log(S.sum_W);
  if (rg.t_min != -DBL_MAX) { *out = log_p_region - log(rg.t_max - rg.t_min); return; }
  const double fa = S.f, lam = S.lambda_X;
  const int m = rg.min_muts;
  const double tS = f.t[S.node_base + f.pos_of_node[S.node_base + rg.branch]];
  const double s_min = fabs(S.t_X - tS);
  const double t_early = fmin(S.t_X, tS);
  const double s_max = s_min + 20.0 * (S.t_max_tip - t_early);
  const double x_min = lam * fa * s_min, x_max = lam * fa * s_max;
  const double sv = S.t_X - t + tS - t;
  if (sv > s_max + 1e-6) { *out = -CUDART_INF; return; }
  if (x_max < 0.01) {
    const double alpha = fa * m + 1;
    *out = log_p_region + 0.6931471805599453 + log(alpha) + (alpha - 1) * log(sv) + -alpha * log(s_max) + -log1p(-pow(s_min / s_max, alpha));
    return;
  }
  const double a = fa * m + 1;
  *out = log_p_region + 0.6931471805599453 + log(lam * fa) + fa * m * log(lam * fa * sv) + -lam * fa * sv + -lgamma(a)
         - log(dev_gamma_q(a, x_min) - dev_gamma_q(a, x_max));
}

// x with Q(a, x) = q: bracket by doubling, then Newton steps safeguarded by bisection (dQ/dx = -x^(a-1) e^-x / Gamma(a))
__device__ double dev_gamma_q_inv(double a, double q) {
  if (q <= 0.0) return CUDART_INF;
  if (q >= 1.0) return 0.0;
  double lo = 0.0, hi = a > 1.0 ? a : 1.0;
  while (dev_gamma_q(a, hi) > q) { lo = hi; hi *= 2.0; if (hi > 1e300) return CUDART_INF; }
  double x = 0.5 * (lo + hi);
  for (int it = 0; it < 400; ++it) {
    const double fv = dev_gamma_q(a, x) - q;
    if (fv > 0.0) lo = x; else hi = x;
    const double dq = -exp((a - 1.0) * log(x) - x - lgamma(a));
    double xn = (dq != 0.0 && isfinite(dq)) ? x - fv / dq : 0.5 * (lo + hi);
    if (!(xn > lo && xn < hi)) xn = 0.5 * (lo + hi);
    if (fabs(xn - x) <= 4e-16 * fabs(x)) { x = xn; break; }
    x = xn;
  }
  return x;
}

// which: 0 -> out[i] = Q(a[i], x[i]);  1 -> out[i] = x with Q(a[i], x) = x_or_q[i]
__global__ void gamma_q_kernel(int which, int n, const double* __restrict__ a, const double* __restrict__ x_or_q, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = which == 0 ? dev_gamma_q(a[i], x_or_q[i]) : dev_gamma_q_inv(a[i], x_or_q[i]);
}

}  // namespace dphy

using namespace dphy;

struct dphy_spr_batch {
  SprBatchDev dev{};
  void* d_block = nullptr;        // one stream-ordered allocation: studies + workspaces + slab
  size_t bytes = 0;
  int32_t num = 0;
  std::vector<SprStudy> host;     // filled by get_summaries
  bool fetched = false;
  SprGroupDev* d_groups = nullptr;
  bool weighted = false;          // spr_weights_kernel + spr_normalize_kernel have run for the current (lambda_X, f, t_max_tip)
  int status = DPHY_OK;           // sticky: the first per-study error found by spr_fetch, returned by every accessor
  std::string status_msg;
  dphy_forest* forest = nullptr;
  // the batch's normalisation pass was put on the ctx's tail stream: ev_done fires when it is through.  Accessors join first.
  cudaEvent_t ev_done = nullptr;
  bool tail_pending = false;
};

// order the main stream after the batch's tail (device-side wait; no host block)
static int spr_join_tail(dphy_ctx* ctx, dphy_spr_batch* b) {
  if (!b->tail_pending) return DPHY_OK;
  DPHY_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, b->ev_done, 0));
  b->tail_pending = false;
  return DPHY_OK;
}

namespace {
// the study-independent tables of the event-scan path: built by the first grouped batch on a forest, freed with it
int ensure_spr_tables(dphy_ctx* ctx, dphy_forest* fo) {
  if (fo->d_spr_eopen) return DPHY_OK;
  const size_t N = (size_t)fo->h.num_nodes, M = (size_t)fo->total_muts;
  int max_nodes = 1;
  for (const TreeDev& T : fo->trees) max_nodes = std::max(max_nodes, T.num_nodes);
  const int max_tiles = (max_nodes + kPmTile - 1) / kPmTile;
  Slab slab;
  const int b_eopen = slab.reserve(sizeof(int32_t) * N), b_tnode = slab.reserve(sizeof(int32_t) * (N + M + 1));
  const int b_ev = slab.reserve(sizeof(int32_t) * (2 * M + 1)), b_pm = slab.reserve(sizeof(int32_t) * N);
  const int b_tt = slab.reserve(sizeof(int32_t) * (size_t)max_tiles * fo->h.num_trees);
  DevBlock blk(ctx->stream);
  if (!blk.alloc(slab.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(spr tables)");
  char* d = blk.p;
  int32_t* pm = slab.at<int32_t>(d, b_pm);
  int32_t* tt = slab.at<int32_t>(d, b_tt);
  spr_tab_pm_kernel<<<dim3(max_tiles, fo->h.num_trees), 1024, 0, ctx->stream>>>(fo->h, pm, tt, max_tiles);
  spr_tab_fill_kernel<<<dim3((max_nodes + 255) / 256, fo->h.num_trees), 256, 0, ctx->stream>>>(fo->h, pm, tt, max_tiles, slab.at<int32_t>(d, b_eopen),
                                                                                             slab.at<int32_t>(d, b_tnode), slab.at<int32_t>(d, b_ev));
  ctx->launches += 2;
  const int st = check_cuda(ctx, cudaGetLastError(), "spr table kernels launch");
  if (st != DPHY_OK) return st;
  fo->allocs.push_back(blk.release());
  fo->bytes += slab.total;
  fo->d_spr_eopen = slab.at<int32_t>(d, b_eopen); fo->d_spr_tnode = slab.at<int32_t>(d, b_tnode); fo->d_spr_ev = slab.at<int32_t>(d, b_ev);
  return DPHY_OK;
}

// dphy_spr_batch_destroy as a deleter: a batch under construction is released by it on every early return
struct BatchDestroy {
  dphy_ctx* ctx;
  void operator()(dphy_spr_batch* b) const { dphy_spr_batch_destroy(ctx, b); }
};
}

extern "C" {

int dphy_spr_study_batch(dphy_ctx* ctx, dphy_forest* fo, int32_t n, const dphy_spr_request* reqs, dphy_spr_batch** out) {
  if (!ctx || !fo || !out || n < 0 || (n > 0 && !reqs)) return DPHY_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  cudaSetDevice(ctx->device);
  int st = refresh_sites(ctx, fo);
  if (st != DPHY_OK) return st;
  std::unique_ptr<dphy_spr_batch, BatchDestroy> b(new (std::nothrow) dphy_spr_batch(), BatchDestroy{ctx});
  if (!b) return DPHY_ERR_OUT_OF_MEMORY;
  b->num = n; b->forest = fo;
  b->host.resize(n);
  int max_tiles = 1, max_tiles256 = 0;
  bool any_frontier = false, any_swept_limited = false;
  int num_bounded = 0;
  for (int i = 0; i < n; ++i) num_bounded += reqs[i].max_muts_from_start != INT_MAX;
  // the batch's slab: per-group and per-study arrays, then the path targets.  Their offsets from b->dev.slab go straight into the
  // group and study records, so a running offset lays them out (a Slab's block records cost measurable host time at 1,024 studies)
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t at = off; off = align_up(off + bytes); return (int64_t)at; };
  std::vector<std::pair<size_t, const void*>> copies;   // (slab offset, host ptr) with sizes below
  std::vector<size_t> copy_bytes;
  // ---- grouping: full (unbounded) studies of the same tree go 32 at a time through the lanes-are-studies kernels ----------------
  constexpr int kMinGroup = 24;     // a group costs the same for 1 or 32 lanes: below ~24 studies the per-study kernels are cheaper
  std::vector<int> group_of(n, -1), lane_of(n, 0);
  std::vector<SprGroupDev> groups;
  std::vector<std::vector<int>> by_tree(fo->h.num_trees);
  for (int i = 0; i < n; ++i)
    if (reqs[i].tree >= 0 && reqs[i].tree < fo->h.num_trees && reqs[i].max_muts_from_start == INT_MAX) by_tree[reqs[i].tree].push_back(i);
  std::vector<int64_t> mut_base(fo->h.num_trees + 1, 0);
  for (int k = 0; k < fo->h.num_trees; ++k) mut_base[k + 1] = mut_base[k] + fo->tree_muts[k];
  for (int k = 0; k < fo->h.num_trees; ++k) {
    const auto& v = by_tree[k];
    for (size_t g0 = 0; g0 < v.size(); g0 += kGroup) {
      if ((int)(v.size() - g0) < kMinGroup) break;       // a thin remainder goes study by study
      SprGroupDev G;
      std::memset(&G, 0, sizeof(G));
      const TreeDev& T = fo->trees[k];
      G.tree = k; G.node_base = T.node_base; G.num_nodes = T.num_nodes; G.L = fo->sites[T.sites_id]->L;
      G.mut_base = (int32_t)mut_base[k];
      G.num = (int32_t)std::min<size_t>(kGroup, v.size() - g0);
      for (int l = 0; l < G.num; ++l) { G.study[l] = v[g0 + l]; group_of[v[g0 + l]] = (int)groups.size(); lane_of[v[g0 + l]] = l; }
      G.off_xT = take((size_t)G.L * kGroup);
      {
        const int64_t M = fo->tree_muts[k];
        if (2 * M + 1 + kEvChunk > INT_MAX || (int64_t)T.num_nodes + M + 64 > INT_MAX) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "spr: tree too large");
        G.num_muts = (int32_t)M; G.num_templates = (int32_t)(T.num_nodes + M);
        G.num_ev_chunks = (int32_t)(2 * M / kEvChunk + 1);           // rows 0 .. 2M
        G.num_t_chunks = (G.num_templates + 31) / 32;                // + one empty chunk, so that KB(N) always has a row
        G.off_S = take((size_t)G.num_ev_chunks * kEvChunk * kGroup);
        G.off_aggS = take(sizeof(int32_t) * ((size_t)G.num_ev_chunks + 1) * kGroup);
        G.off_mask = take(sizeof(uint32_t) * ((size_t)G.num_t_chunks + 1) * kGroup);
        G.off_aggK = take(sizeof(int32_t) * ((size_t)G.num_t_chunks + 2) * kGroup);
        G.off_cbase = take(sizeof(int2) * ((size_t)G.num_t_chunks + 1) * kGroup);
        G.off_consts = take(32 * kGroup + sizeof(int32_t) * kGroup);      // G2Const [32] + root_keep [32]
        G.off_outs = take(64 * kGroup);
        if (g0 == 0) {
          G.trec_owner = 1; G.off_trec = take(48 * (size_t)G.num_templates);
          G.off_csort = take(sizeof(double) * 32 * ((size_t)G.num_t_chunks + 1));
          G.off_cpm = take(sizeof(uint32_t) * 32 * ((size_t)G.num_t_chunks + 1));
          G.off_cq = take(sizeof(int2) * ((size_t)G.num_t_chunks + 1));
        } else {
          const SprGroupDev& G0 = groups[groups.size() - g0 / kGroup];
          G.trec_owner = 0; G.off_trec = G0.off_trec; G.off_csort = G0.off_csort; G.off_cpm = G0.off_cpm; G.off_cq = G0.off_cq;
        }
      }
      groups.push_back(G);
    }
  }
  // (raw log-weights inside the grouped emit were measured slower than the dense weights pass over the stored heads: the two logs
  // per region then run at the emit's ~45 % lane utilisation and low occupancy, 1.26 ms vs 0.68 + 0.23 ms per 128 studies)
  // The event-scan emit computes the raw log-weights itself
  for (int i = 0; i < n; ++i) {
    const dphy_spr_request& r = reqs[i];
    SprStudy& S = b->host[i];
    std::memset(&S, 0, sizeof(S));
    if (r.tree < 0 || r.tree >= fo->h.num_trees) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "spr: tree index out of range");
    const TreeDev& T = fo->trees[r.tree];
    const int L = fo->sites[T.sites_id]->L;
    if (r.X < -1 || r.X >= T.num_nodes) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "spr: X out of range");
    if (r.X == T.root_id) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "spr: X must not be the root (CHECK_NE(X, tree->root))");
    if (r.start_branch < 0 || r.start_branch >= T.num_nodes) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "spr: start branch out of range");
    if (r.start_branch == r.X) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "spr: start region is on branch X");
    if (!(r.lambda_X >= 0.0)) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "spr: lambda_X must be >= 0 (0: enumerate only)");
    if (r.x_state_mode < DPHY_SPR_X_FROM_TREE || r.x_state_mode > DPHY_SPR_X_REL_START) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "spr: unknown x_state_mode");
    if ((r.x_state_mode != DPHY_SPR_X_FROM_TREE || r.X < 0) && ((r.n_x_deltas > 0 && (!r.x_delta_site || !r.x_delta_to)) || (r.n_x_missing > 0 && (!r.x_missing_start || !r.x_missing_end)) || r.n_x_deltas < 0 || r.n_x_missing < 0))
      return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "spr: explicit X state without its arrays");
    S.tree = r.tree; S.X = r.X; S.start_branch = r.start_branch; S.start_mut_idx = r.start_mut_idx;
    S.init_min_muts = r.init_min_muts; S.limit = r.max_muts_from_start; S.can_change_root = r.can_change_root != 0;
    S.t_X = r.t_X; S.lambda_X = r.lambda_X; S.f = r.annealing_factor; S.t_max_tip = r.t_max_tip;
    S.x_mode = (r.X < 0 && r.x_state_mode == DPHY_SPR_X_FROM_TREE) ? DPHY_SPR_X_REL_REF : r.x_state_mode;   // a detached X has no state in the tree
    const bool explicit_x = S.x_mode != DPHY_SPR_X_FROM_TREE;
    S.n_x_deltas = explicit_x ? r.n_x_deltas : 0; S.n_x_missing = explicit_x ? r.n_x_missing : 0;
    for (int k = 0; k < S.n_x_deltas; ++k)
      if (r.x_delta_site[k] < 0 || r.x_delta_site[k] >= L || r.x_delta_to[k] > 3) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "spr: X delta out of range");
    for (int k = 0; k < S.n_x_missing; ++k)
      if (r.x_missing_start[k] < 0 || r.x_missing_end[k] > L || r.x_missing_start[k] >= r.x_missing_end[k]) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "spr: X missing interval out of range");
    const int N = T.num_nodes;
    const bool grouped = group_of[i] >= 0;
    // bounded studies of a small radius walk their ball (kernels_spr_frontier.cuh), the others take the per-study sweeps.
    // Measured on a 100k-tip tree (tools/spr_bounded_timing.py): radius 1: 7.0 vs 9.7 us per study in a batch of 64, 3.4 vs 7.9 in a
    // batch of 512; radius 2: 17.4 vs 9.7 (64), 5.0 vs 7.9 (512) -- a walk lasts as long as its largest ball (mutation-free clades make
    // the ball sizes heavy-tailed) while the sweeps cost the same for every study, so larger radii only walk in large batches.
    constexpr int kFrontierMaxRadius = 4;
    const bool frontier = !grouped && r.max_muts_from_start != INT_MAX && r.max_muts_from_start <= kFrontierMaxRadius &&
                          (r.max_muts_from_start <= 1 || num_bounded >= 256);
    any_frontier |= frontier;
    any_swept_limited |= !grouped && !frontier && r.max_muts_from_start != INT_MAX;
    S.h_stride = grouped ? kGroup : (frontier ? 0 : 1); S.tile_shift = grouped ? 5 : 8;
    S.num_htiles = grouped ? 1 : T.num_tiles;
    if (grouped) {
      const SprGroupDev& G = groups[group_of[i]];
      S.g2 = 1; S.g2_lane = lane_of[i]; S.g2_mut_base = G.mut_base; S.g2_num_templates = G.num_templates;
      S.off_g2S = G.off_S; S.off_g2aggS = G.off_aggS; S.off_g2mask = G.off_mask; S.off_g2aggK = G.off_aggK;
    }
    S.weights_fused = (grouped && r.lambda_X > 0.0) ? 1 : 0;
    max_tiles = std::max(max_tiles, S.num_htiles);
    if (!grouped && !frontier) max_tiles256 = std::max(max_tiles256, T.num_tiles);
    // exact upper bound on regions: every non-root node has n+1 regions, the root has 1
    const int64_t cap64 = (int64_t)N + fo->tree_muts[r.tree] + 1;
    if (cap64 > INT_MAX) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "spr: region capacity overflow");
    S.region_cap = (int32_t)cap64;
    S.path_cap = fo->tree_max_depth[r.tree] + 2;
    S.off_xtab = take(L);
    S.off_xkey = take(sizeof(uint32_t) * (size_t)L);
    S.off_path = take(sizeof(int32_t) * S.path_cap);
    S.off_xpath = take(sizeof(int32_t) * S.path_cap);
    S.off_pae = take(sizeof(int2) * S.path_cap);
    if (grouped) {
      S.off_H = 0; S.off_C = 0; S.off_KB = 0;          // unused: H and KB are read off the group's event rows / keep masks
    } else {
      S.off_H = take(sizeof(int32_t) * N);
      S.off_C = take(sizeof(int32_t) * N);
      S.off_KB = take(sizeof(int32_t) * (N + 1));
    }
    S.off_seg = take(sizeof(int32_t) * kSegStride * (size_t)S.path_cap);
    S.off_hang = grouped ? take(sizeof(int32_t) * (size_t)S.path_cap) : (int64_t)off;
    // chunks that straddle a segment boundary of the study: at most two per path node
    S.hmix_cap = grouped ? 2 * S.path_cap + 2 : 0;
    S.off_hmix = take(sizeof(int32_t) * 32 * (size_t)S.hmix_cap);
    S.off_part = take(sizeof(double) * kNormBlocks);
    S.off_tj = take(sizeof(int2) * (size_t)T.num_tiles);       // classify() of the first / last node of every tile
    S.off_xd_site = take(sizeof(int32_t) * std::max(1, S.n_x_deltas));
    S.off_xd_to = take(std::max(1, S.n_x_deltas));
    S.off_xm_start = take(sizeof(int32_t) * std::max(1, S.n_x_missing));
    S.off_xm_end = take(sizeof(int32_t) * std::max(1, S.n_x_missing));
    S.off_regions = take(sizeof(RegionHead) * (size_t)S.region_cap);
    S.off_nw = take(sizeof(double2) * (size_t)S.region_cap);
    S.off_lw = take(sizeof(double) * (size_t)S.region_cap);     // raw log-weights between emit and normalise
    if (S.n_x_deltas) {
      copies.push_back({(size_t)S.off_xd_site, r.x_delta_site}); copy_bytes.push_back(sizeof(int32_t) * S.n_x_deltas);
      copies.push_back({(size_t)S.off_xd_to, r.x_delta_to}); copy_bytes.push_back(S.n_x_deltas);
    }
    if (S.n_x_missing) {
      copies.push_back({(size_t)S.off_xm_start, r.x_missing_start}); copy_bytes.push_back(sizeof(int32_t) * S.n_x_missing);
      copies.push_back({(size_t)S.off_xm_end, r.x_missing_end}); copy_bytes.push_back(sizeof(int32_t) * S.n_x_missing);
    }
  }
  // path targets: studies grouped by tree, two targets (start node, X) per study, sorted per tree on the device
  std::vector<int32_t> path_order(n);
  std::vector<SprPathTree> path_trees;
  {
    std::vector<std::vector<int32_t>> by(fo->h.num_trees);
    for (int i = 0; i < n; ++i) by[reqs[i].tree].push_back(i);
    int32_t first = 0;
    for (int k = 0; k < fo->h.num_trees; ++k) {
      if (by[k].empty()) continue;
      std::copy(by[k].begin(), by[k].end(), path_order.begin() + first);
      path_trees.push_back(SprPathTree{k, first, (int32_t)by[k].size(), 0});
      first += (int32_t)by[k].size();
    }
  }
  const size_t off_porder = take(sizeof(int32_t) * std::max(1, n));
  const size_t off_ptrees = take(sizeof(SprPathTree) * std::max<size_t>(1, path_trees.size()));
  const size_t off_traw = take(sizeof(int32_t) * 2 * std::max(1, n));
  const size_t off_tgt = take(sizeof(SprPathTarget) * 2 * std::max(1, n));
  const size_t off_taux = take(sizeof(SprPathTargetAux) * 2 * std::max(1, n));
  if (n > 0) {
    copies.push_back({off_porder, path_order.data()}); copy_bytes.push_back(sizeof(int32_t) * n);
    copies.push_back({off_ptrees, path_trees.data()}); copy_bytes.push_back(sizeof(SprPathTree) * path_trees.size());
  }
  // the block: studies, look-back workspaces, flags + tickets, groups, then the slab
  Slab hdr;
  const int b_studies = hdr.reserve(sizeof(SprStudy) * std::max(1, n));
  const int b_agg = hdr.reserve(sizeof(int32_t) * 3 * ((size_t)max_tiles + 1) * std::max(1, n));
  const int b_flag = hdr.reserve(256), b_ticket = hdr.reserve(sizeof(uint32_t) * 4 * std::max(1, n));
  const int b_groups = hdr.reserve(sizeof(SprGroupDev) * std::max<size_t>(1, groups.size()));
  const size_t total = hdr.total + off;
  char* d = nullptr;
  size_t block_bytes = total;
  // a block left by an earlier batch (see dphy_ctx::spr_blocks): the oldest one that is large enough, once two are waiting
  if (ctx->spr_blocks.size() >= 2) {
    for (size_t i = 0; i < ctx->spr_blocks.size(); ++i) {
      dphy_ctx::SprBlock blk = ctx->spr_blocks[i];
      if (blk.bytes < total || blk.bytes > 2 * total + (64u << 20)) continue;
      ctx->spr_blocks.erase(ctx->spr_blocks.begin() + i);
      if (blk.ev) { cudaStreamWaitEvent(ctx->stream, blk.ev, 0); cudaEventDestroy(blk.ev); }
      d = (char*)blk.ptr; block_bytes = blk.bytes;
      break;
    }
  }
  if (!d) {
    DevBlock blk(ctx->stream);
    cudaError_t ce = cudaSuccess;
    if (!blk.alloc(total, &ce)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, std::string("cudaMallocAsync(spr batch): ") + cudaGetErrorString(ce));
    d = blk.release();
  }
  b->d_block = d; b->bytes = block_bytes;     // from here on freed (or parked) by dphy_spr_batch_destroy
  b->dev.studies = hdr.at<SprStudy>(d, b_studies);
  b->dev.tile_agg = hdr.at<int32_t>(d, b_agg);
  b->dev.tile_flag = hdr.at<uint32_t>(d, b_flag);
  b->dev.ticket = hdr.at<uint32_t>(d, b_ticket);
  b->dev.slab = d + hdr.total;
  b->dev.num_studies = n; b->dev.max_tiles = max_tiles;
  b->dev.g2_eopen = nullptr; b->dev.g2_tnode = nullptr; b->dev.g2_ev = nullptr; b->dev.g2_mut_off = fo->h.mut_off;
  if (!groups.empty()) {
    st = ensure_spr_tables(ctx, fo);
    if (st != DPHY_OK) return st;
    b->dev.g2_eopen = fo->d_spr_eopen; b->dev.g2_tnode = fo->d_spr_tnode; b->dev.g2_ev = fo->d_spr_ev;
  }
  b->d_groups = hdr.at<SprGroupDev>(d, b_groups);
  if (n == 0) { *out = b.release(); return DPHY_OK; }
  // flags + tickets start at zero; studies + X overlays uploaded through the pinned staging buffer
  cudaError_t ce = cudaMemsetAsync(hdr.at<char>(d, b_flag), 0, hdr.blocks[b_groups].off - hdr.blocks[b_flag].off, ctx->stream);
  size_t stage = sizeof(SprStudy) * n + align_up(sizeof(SprGroupDev) * groups.size());
  for (size_t cb : copy_bytes) stage += align_up(cb);
  if (ce == cudaSuccess) {
    PinnedStage pin(ctx, stage);
    if (pin.status != DPHY_OK) return pin.status;
    char* hb = pin.p;
    std::memcpy(hb, b->host.data(), sizeof(SprStudy) * n);
    ce = cudaMemcpyAsync(b->dev.studies, hb, sizeof(SprStudy) * n, cudaMemcpyHostToDevice, ctx->stream);
    size_t so = sizeof(SprStudy) * n;
    if (!groups.empty() && ce == cudaSuccess) {
      std::memcpy(hb + so, groups.data(), sizeof(SprGroupDev) * groups.size());
      ce = cudaMemcpyAsync(b->d_groups, hb + so, sizeof(SprGroupDev) * groups.size(), cudaMemcpyHostToDevice, ctx->stream);
      so += align_up(sizeof(SprGroupDev) * groups.size());
    }
    for (size_t k = 0; k < copies.size() && ce == cudaSuccess; ++k) {
      std::memcpy(hb + so, copies[k].second, copy_bytes[k]);
      ce = cudaMemcpyAsync(b->dev.slab + copies[k].first, hb + so, copy_bytes[k], cudaMemcpyHostToDevice, ctx->stream);
      so += align_up(copy_bytes[k]);
    }
  }
  if (ce != cudaSuccess) return check_cuda(ctx, ce, "spr batch upload");
  int max_nodes = 1, group_L = 1;
  for (int i = 0; i < n; ++i) max_nodes = std::max(max_nodes, fo->trees[reqs[i].tree].num_nodes);
  for (const SprGroupDev& G : groups) group_L = std::max(group_L, G.L);
  const int ng = (int)groups.size();
  const bool any_single = max_tiles256 > 0;        // studies on the per-study path
  {
    char* sl = b->dev.slab;
    const SprPathTree* d_pt = (const SprPathTree*)(sl + off_ptrees);
    spr_init_kernel<<<(unsigned)path_trees.size(), 256, 0, ctx->stream>>>(fo->h, b->dev, d_pt, (const int32_t*)(sl + off_porder), (int32_t*)(sl + off_traw),
                                                                         (SprPathTarget*)(sl + off_tgt), (SprPathTargetAux*)(sl + off_taux));
    // fork: what depends on the tree and the studies' positions alone (constants, template records, keep masks) runs on the side stream
    // while the main stream walks the latency-bound chain paths -> X tables -> event scan
    if (ng > 0) {
      if (!ctx->aux_stream) {
        if (cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming) != cudaSuccess) {
          return set_error(ctx, DPHY_ERR_CUDA, "spr: side stream");
        }
      }
      cudaEventRecord(ctx->ev_fork, ctx->stream);
      cudaStreamWaitEvent(ctx->aux_stream, ctx->ev_fork, 0);
    }
    spr_paths_kernel<<<dim3((max_nodes + kSetupThreads - 1) / kSetupThreads, (unsigned)path_trees.size()), kSetupThreads, 0, ctx->stream>>>(
        fo->h, b->dev, d_pt, (const SprPathTarget*)(sl + off_tgt), (const SprPathTargetAux*)(sl + off_taux));
  }
  spr_xtab_kernel<<<dim3(kXtabSlices, n), kSetupThreads, 0, ctx->stream>>>(fo->h, b->dev);
  int launched = 3;
  const dim3 grid_scan((std::max(max_tiles256, 1) + kScanSub - 1) / kScanSub, n);
  if (any_single) { spr_scan_kernel<0><<<grid_scan, kTile, 0, ctx->stream>>>(fo->h, b->dev); ++launched; }
  int g2_ev_chunks = 0, g2_t_chunks = 0, g2_templates = 1;
  for (const SprGroupDev& G : groups) {
    g2_ev_chunks = std::max(g2_ev_chunks, G.num_ev_chunks); g2_t_chunks = std::max(g2_t_chunks, G.num_t_chunks + 1);
    g2_templates = std::max(g2_templates, G.num_templates);
  }
  const dim3 grid_g2t((g2_t_chunks + kG2Warps - 1) / kG2Warps, std::max(ng, 1));
  if (ng > 0) {
    cudaStream_t side = ctx->aux_stream;
    spr_xT_kernel<<<dim3((group_L + 255) / 256, ng), 256, 0, ctx->stream>>>(b->dev, b->d_groups);
    spr_g2_consts_kernel<<<ng, kGroup, 0, side>>>(fo->h, b->dev, b->d_groups);
    spr_g2_templ_kernel<<<dim3((g2_t_chunks * 32 + 255) / 256, ng), 256, 0, side>>>(fo->h, b->dev, b->d_groups);
    launched += 2;
    spr_g2_count_kernel<<<dim3((g2_t_chunks + kCountWarps * kCountPerWarp - 1) / (kCountWarps * kCountPerWarp), ng), kCountWarps * 32, 0, side>>>(fo->h, b->dev, b->d_groups);
    spr_g2_prefix_kernel<<<dim3(kPfxCtas, ng), 1024, 0, side>>>(b->dev, b->d_groups, 1);
    spr_g2_scan_kernel<<<dim3((g2_ev_chunks + kG2Warps - 1) / kG2Warps, ng), kG2Warps * 32, 0, ctx->stream>>>(fo->h, b->dev, b->d_groups);
    spr_g2_prefix_kernel<<<dim3(kPfxCtas, ng), 1024, 0, ctx->stream>>>(b->dev, b->d_groups, 0);
    cudaEventRecord(ctx->ev_join, ctx->aux_stream);
    cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0);
    launched += 5;
  }
  if (any_frontier) { spr_frontier_kernel<<<(n + 3) / 4, 128, 0, ctx->stream>>>(fo->h, b->dev); ++launched; }
  if (any_swept_limited) {
    spr_tile_prefix_kernel<<<n, kSetupThreads, 0, ctx->stream>>>(fo->h, b->dev);
    spr_scan_kernel<1><<<grid_scan, kTile, 0, ctx->stream>>>(fo->h, b->dev);
    launched += 2;
  }
  spr_segments_kernel<<<n, kSetupThreads, 0, ctx->stream>>>(fo->h, b->dev);
  ++launched;
  if (any_single) {
    const dim3 grid_emit((max_tiles256 + kEmitSub - 1) / kEmitSub, n);
    spr_emit_kernel<<<grid_emit, kTile, 0, ctx->stream>>>(fo->h, b->dev);
    ++launched;
  }
  bool any_weighted = false, any_unfused = false;
  for (int i = 0; i < n; ++i) {
    any_weighted |= b->host[i].lambda_X > 0.0;
    any_unfused |= b->host[i].lambda_X > 0.0 && !b->host[i].weights_fused;
  }
  const bool g2_emit = ng > 0;
  if (g2_emit) { spr_g2_bases_kernel<<<dim3(kGroup, ng, kBasesSlices), kBasesThreads, 0, ctx->stream>>>(b->dev, b->d_groups); ++launched; }
  // The bulk passes of a batch -- the template emit (heads + raw log-weights: issue- and bandwidth-bound), the dense weights pass if
  // any, the normalisation (bandwidth-bound) -- read the forest and write only the batch's own block: they go to the TAIL stream, so
  // that the set-up chain of the NEXT batch (paths, X tables, event scan, segments, bases: latency-bound kernels with small grids,
  // on the higher-priority main stream) runs next to them.  Every accessor of the batch, and every entry point that edits or frees
  // the forest, joins the tail first.
  const bool use_tail = g2_emit || any_weighted;
  if (use_tail) {
    if (!ctx->tail_stream) {
      if (cudaStreamCreateWithFlags(&ctx->tail_stream, cudaStreamNonBlocking) != cudaSuccess ||
          cudaEventCreateWithFlags(&ctx->ev_tail, cudaEventDisableTiming) != cudaSuccess)
        return set_error(ctx, DPHY_ERR_CUDA, "spr: tail stream");
    }
    if (cudaEventCreateWithFlags(&b->ev_done, cudaEventDisableTiming) != cudaSuccess) return set_error(ctx, DPHY_ERR_CUDA, "spr: tail event");
    cudaEventRecord(ctx->ev_tail, ctx->stream);
    cudaStreamWaitEvent(ctx->tail_stream, ctx->ev_tail, 0);
  }
  cudaStream_t ts = use_tail ? ctx->tail_stream : ctx->stream;
  if (g2_emit) {
    spr_g2_emit_kernel<<<grid_g2t, kG2Warps * 32, 0, ts>>>(fo->h, b->dev, b->d_groups);
    ++launched;
  }
  if (any_weighted) {
    if (any_unfused) { spr_weights_kernel<<<dim3(kWeightBlocks, n), 256, 0, ts>>>(fo->h, b->dev); ++launched; }
    spr_normalize_kernel<<<dim3(kNormBlocks, n), 256, 0, ts>>>(b->dev);
    ++launched;
    b->weighted = true;
  }
  if (use_tail) { cudaEventRecord(b->ev_done, ctx->tail_stream); b->tail_pending = true; ctx->tail_dirty = true; }
  ctx->launches += launched;
  st = check_cuda(ctx, cudaGetLastError(), "spr kernels launch");
  if (st != DPHY_OK) return st;
  *out = b.release();
  return DPHY_OK;
}

void dphy_spr_batch_destroy(dphy_ctx* ctx, dphy_spr_batch* b) {
  if (!b) return;
  if (ctx && b->d_block) {
    cudaSetDevice(ctx->device);
    if (b->tail_pending && ctx->tail_stream) {
      // the tail may still be running: the block is parked with the tail's event (the main stream does not wait, so the next
      // batch's set-up proceeds) and handed to a later batch; the oldest parked block is released when too many are waiting
      ctx->spr_blocks.push_back({b->d_block, b->bytes, b->ev_done});
      b->ev_done = nullptr;
      while (ctx->spr_blocks.size() > dphy_ctx::kSprBlocksKept) {
        dphy_ctx::SprBlock old = ctx->spr_blocks.front();
        ctx->spr_blocks.erase(ctx->spr_blocks.begin());
        if (old.ev) { cudaStreamWaitEvent(ctx->stream, old.ev, 0); cudaEventDestroy(old.ev); }
        cudaFreeAsync(old.ptr, ctx->stream);
      }
    } else {
      cudaFreeAsync(b->d_block, ctx->stream);
    }
  }
  if (b->ev_done) cudaEventDestroy(b->ev_done);
  delete b;
}

static int spr_fetch(dphy_ctx* ctx, dphy_spr_batch* b) {
  if (b->status != DPHY_OK) return set_error(ctx, b->status, b->status_msg);
  { const int js = spr_join_tail(ctx, b); if (js != DPHY_OK) return js; }
  if (b->fetched || b->num == 0) return DPHY_OK;
  DPHY_CUDA(ctx, cudaMemcpyAsync(b->host.data(), b->dev.studies, sizeof(SprStudy) * b->num, cudaMemcpyDeviceToHost, ctx->stream));
  DPHY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  b->fetched = true;
  for (int i = 0; i < b->num; ++i) {
    const char* what = nullptr; int st = DPHY_OK;
    if (b->host[i].error == kSprErrXNoParent) { st = DPHY_ERR_INVALID_ARGUMENT; what = "X has no parent"; }
    else if (b->host[i].error == kSprErrStartMutIdx) { st = DPHY_ERR_OUT_OF_RANGE; what = "start_mut_idx out of range for the start branch"; }
    else if (b->host[i].error == kSprErrStartInXSubtree) { st = DPHY_ERR_INVALID_ARGUMENT; what = "start region lies inside X's subtree"; }
    else if (b->host[i].error == kSprErrPathMuts) { st = DPHY_ERR_INTERNAL; what = "more than 2^28 mutations on the root path"; }
    else if (b->host[i].error == kSprErrFrontierCap) { st = DPHY_ERR_INTERNAL; what = "the bounded-radius walk found more regions than the study's region capacity"; }
    else if (b->host[i].error == kSprErrHmixCap) { st = DPHY_ERR_INTERNAL; what = "more template chunks straddle the study's path segments than the grouped emit has offset rows for"; }
    else if (b->host[i].total_regions > b->host[i].region_cap) { st = DPHY_ERR_INTERNAL; what = "region capacity exceeded"; }
    if (st != DPHY_OK) {
      // sticky: every later accessor of this batch (getters, pick, find) reports the same failure, naming the request
      b->status = st;
      b->status_msg = "spr: request " + std::to_string(i) + ": " + what;
      return set_error(ctx, b->status, b->status_msg);
    }
  }
  return DPHY_OK;
}

int dphy_spr_batch_get_summaries(dphy_ctx* ctx, dphy_spr_batch* b, dphy_spr_summary* out) {
  if (!ctx || !b || !out) return DPHY_ERR_INVALID_ARGUMENT;
  int st = spr_fetch(ctx, b);
  if (st != DPHY_OK) return st;
  int64_t off = 0;
  for (int i = 0; i < b->num; ++i) {
    const SprStudy& S = b->host[i];
    out[i].mu = S.mu; out[i].log_Wmax = S.log_Wmax; out[i].sum_W_over_Wmax = S.sum_W;
    out[i].num_regions = S.total_regions; out[i].num_missing_at_X = S.num_missing; out[i].region_offset = off;
    off += S.total_regions;
  }
  return DPHY_OK;
}

int64_t dphy_spr_batch_total_regions(dphy_ctx* ctx, dphy_spr_batch* b) {
  if (!ctx || !b) return DPHY_ERR_INVALID_ARGUMENT;
  int st = spr_fetch(ctx, b);
  if (st != DPHY_OK) return st;
  int64_t tot = 0;
  for (int i = 0; i < b->num; ++i) tot += b->host[i].total_regions;
  return tot;
}

int64_t dphy_spr_batch_get_regions(dphy_ctx* ctx, dphy_spr_batch* b, int32_t request, dphy_candidate_region* out, int64_t cap) {
  if (!ctx || !b || (!out && cap > 0) || request >= b->num) return DPHY_ERR_INVALID_ARGUMENT;
  int st = spr_fetch(ctx, b);
  if (st != DPHY_OK) return st;
  int64_t w = 0;
  const int lo = request < 0 ? 0 : request, hi = request < 0 ? b->num : request + 1;
  for (int i = lo; i < hi; ++i) {
    const SprStudy& S = b->host[i];
    if (w + S.total_regions > cap) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "spr: output capacity too small");
    if (S.total_regions > 0) {
      // head and tail arrays -> the reference's 48-byte records, interleaved by two strided copies
      char* dst = reinterpret_cast<char*>(out + w);
      DPHY_CUDA(ctx, cudaMemcpy2DAsync(dst, sizeof(dphy_candidate_region), b->dev.slab + S.off_regions, sizeof(RegionHead), sizeof(RegionHead),
                                       (size_t)S.total_regions, cudaMemcpyDeviceToHost, ctx->stream));
      if (b->weighted && S.lambda_X > 0.0) {
        DPHY_CUDA(ctx, cudaMemcpy2DAsync(dst + offsetof(dphy_candidate_region, log_W_over_Wmax), sizeof(dphy_candidate_region),
                                         b->dev.slab + S.off_nw, sizeof(double2), sizeof(double2), (size_t)S.total_regions,
                                         cudaMemcpyDeviceToHost, ctx->stream));
      } else {
        // enumerate-only study: the reference's builder leaves both weights at 0.0 (core/spr_study.h:26-27)
        for (int64_t k = 0; k < S.total_regions; ++k) { out[w + k].log_W_over_Wmax = 0.0; out[w + k].W_over_Wmax = 0.0; }
      }
    }
    w += S.total_regions;
  }
  DPHY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return w;
}

int dphy_spr_batch_set_weights(dphy_ctx* ctx, dphy_spr_batch* b, const dphy_spr_weight_params* params) {
  if (!ctx || !b || (!params && b->num > 0)) return DPHY_ERR_INVALID_ARGUMENT;
  if (b->status != DPHY_OK) return set_error(ctx, b->status, b->status_msg);
  if (b->num == 0) return DPHY_OK;
  cudaSetDevice(ctx->device);
  { const int js = spr_join_tail(ctx, b); if (js != DPHY_OK) return js; }
  for (int i = 0; i < b->num; ++i)
    if (!(params[i].lambda_X > 0.0)) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "spr: lambda_X must be > 0");
  PinnedStage pin(ctx, sizeof(double) * 3 * b->num);
  if (pin.status != DPHY_OK) return pin.status;
  double* hb = reinterpret_cast<double*>(pin.p);
  for (int i = 0; i < b->num; ++i) { hb[3 * i] = params[i].lambda_X; hb[3 * i + 1] = params[i].annealing_factor; hb[3 * i + 2] = params[i].t_max_tip; }
  const size_t mark = ctx->arena.mark();
  double* d_wp = (double*)ctx->arena.alloc(sizeof(double) * 3 * b->num);
  if (!d_wp) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "arena exhausted (spr weights)");
  cudaError_t ce = cudaMemcpyAsync(d_wp, hb, sizeof(double) * 3 * b->num, cudaMemcpyHostToDevice, ctx->stream);
  pin.reset();
  if (ce == cudaSuccess) {
    spr_set_weight_params_kernel<<<(b->num + 127) / 128, 128, 0, ctx->stream>>>(b->forest->h, b->dev, d_wp);
    spr_weights_kernel<<<dim3(kWeightBlocks, b->num), 256, 0, ctx->stream>>>(b->forest->h, b->dev);
    spr_normalize_kernel<<<dim3(kNormBlocks, b->num), 256, 0, ctx->stream>>>(b->dev);
    ctx->launches += 3;
    ce = cudaGetLastError();
  }
  ctx->arena.release(mark);
  if (ce != cudaSuccess) return check_cuda(ctx, ce, "spr set_weights");
  b->weighted = true;
  b->fetched = false;       // summaries (mu, log_Wmax, sum_W) changed
  return DPHY_OK;
}

int64_t dphy_spr_batch_get_region_weights(dphy_ctx* ctx, dphy_spr_batch* b, int32_t request, dphy_candidate_region* out, int64_t cap) {
  if (!ctx || !b || (!out && cap > 0) || request >= b->num) return DPHY_ERR_INVALID_ARGUMENT;
  int st = spr_fetch(ctx, b);
  if (st != DPHY_OK) return st;
  if (!b->weighted) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "spr: this batch has no weights (lambda_X == 0 and dphy_spr_batch_set_weights not called)");
  int64_t w = 0;
  const int lo = request < 0 ? 0 : request, hi = request < 0 ? b->num : request + 1;
  for (int i = lo; i < hi; ++i) {
    const SprStudy& S = b->host[i];
    if (w + S.total_regions > cap) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "spr: output capacity too small");
    if (S.total_regions > 0)
      DPHY_CUDA(ctx, cudaMemcpy2DAsync(reinterpret_cast<char*>(out + w) + offsetof(dphy_candidate_region, log_W_over_Wmax), sizeof(dphy_candidate_region),
                                       b->dev.slab + S.off_nw, sizeof(double2), sizeof(double2), (size_t)S.total_regions,
                                       cudaMemcpyDeviceToHost, ctx->stream));
    w += S.total_regions;
  }
  DPHY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return w;
}

int dphy_spr_batch_pick_nexus_regions(dphy_ctx* ctx, dphy_spr_batch* b, const double* r, int32_t* out_idx) {
  if (!ctx || !b || !r || !out_idx) return DPHY_ERR_INVALID_ARGUMENT;
  if (b->num == 0) return DPHY_OK;
  { const int st0 = spr_fetch(ctx, b); if (st0 != DPHY_OK) return st0; }
  if (!b->weighted) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "spr: this batch has no weights");
  const size_t mark = ctx->arena.mark();
  double* d_r = (double*)ctx->arena.alloc(sizeof(double) * b->num);
  int32_t* d_o = (int32_t*)ctx->arena.alloc(sizeof(int32_t) * b->num);
  if (!d_r || !d_o) { ctx->arena.release(mark); return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "arena exhausted (spr pick)"); }
  DPHY_CUDA(ctx, cudaMemcpyAsync(d_r, r, sizeof(double) * b->num, cudaMemcpyHostToDevice, ctx->stream));
  spr_pick_kernel<<<(b->num + 3) / 4, 128, 0, ctx->stream>>>(b->dev, d_r, d_o);
  ctx->launches += 1;
  int st = check_cuda(ctx, cudaGetLastError(), "spr_pick_kernel");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaMemcpyAsync(out_idx, d_o, sizeof(int32_t) * b->num, cudaMemcpyDeviceToHost, ctx->stream), "D2H");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "spr pick");
  ctx->arena.release(mark);
  return st;
}

int dphy_spr_batch_find_region(dphy_ctx* ctx, dphy_spr_batch* b, int32_t request, int32_t branch, double t, int32_t* out_idx) {
  if (!ctx || !b || !out_idx || request < 0 || request >= b->num) return DPHY_ERR_INVALID_ARGUMENT;
  { const int st0 = spr_fetch(ctx, b); if (st0 != DPHY_OK) return st0; }
  const size_t mark = ctx->arena.mark();
  int32_t* d_o = (int32_t*)ctx->arena.alloc(sizeof(int32_t));
  if (!d_o) { ctx->arena.release(mark); return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "arena exhausted (spr find)"); }
  const int32_t init = INT_MAX;
  DPHY_CUDA(ctx, cudaMemcpyAsync(d_o, &init, sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
  spr_find_kernel<<<64, 256, 0, ctx->stream>>>(b->dev, request, branch, t, d_o);
  ctx->launches += 1;
  int32_t res = INT_MAX;
  int st = check_cuda(ctx, cudaGetLastError(), "spr_find_kernel");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaMemcpyAsync(&res, d_o, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream), "D2H");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "spr find");
  ctx->arena.release(mark);
  *out_idx = res == INT_MAX ? -1 : res;
  return st;
}

int dphy_spr_batch_log_alpha_in_region(dphy_ctx* ctx, dphy_spr_batch* b, int32_t request, int32_t region_idx, double t, double* out) {
  if (!ctx || !b || !out || request < 0 || request >= b->num) return DPHY_ERR_INVALID_ARGUMENT;
  { const int st0 = spr_fetch(ctx, b); if (st0 != DPHY_OK) return st0; }
  if (!b->weighted) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "spr: this batch has no weights");
  if (region_idx < 0 || region_idx >= b->host[request].total_regions) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "spr: region index out of range");
  cudaSetDevice(ctx->device);
  const size_t mark = ctx->arena.mark();
  double* d_o = (double*)ctx->arena.alloc(sizeof(double));
  if (!d_o) { ctx->arena.release(mark); return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "arena exhausted (spr log_alpha)"); }
  spr_log_alpha_kernel<<<1, 1, 0, ctx->stream>>>(b->forest->h, b->dev, request, region_idx, t, d_o);
  ctx->launches += 1;
  int st = check_cuda(ctx, cudaGetLastError(), "spr_log_alpha_kernel");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaMemcpyAsync(out, d_o, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream), "D2H");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "spr log_alpha");
  ctx->arena.release(mark);
  return st;
}

static int gamma_q_call(dphy_ctx* ctx, int which, int32_t n, const double* a, const double* v, double* out) {
  if (!ctx || n < 0 || (n > 0 && (!a || !v || !out))) return DPHY_ERR_INVALID_ARGUMENT;
  if (n == 0) return DPHY_OK;
  for (int i = 0; i < n; ++i) {
    if (!(a[i] > 0.0)) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "gamma_q: a must be > 0");
    if (which == 0 ? !(v[i] >= 0.0) : !(v[i] >= 0.0 && v[i] <= 1.0)) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, which == 0 ? "gamma_q: x must be >= 0" : "gamma_q_inv: q must be in [0, 1]");
  }
  cudaSetDevice(ctx->device);
  const size_t mark = ctx->arena.mark();
  double* d = (double*)ctx->arena.alloc(sizeof(double) * 3 * (size_t)n);
  if (!d) { ctx->arena.release(mark); return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "arena exhausted (gamma_q)"); }
  int st = check_cuda(ctx, cudaMemcpyAsync(d, a, sizeof(double) * n, cudaMemcpyHostToDevice, ctx->stream), "H2D");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaMemcpyAsync(d + n, v, sizeof(double) * n, cudaMemcpyHostToDevice, ctx->stream), "H2D");
  if (st == DPHY_OK) {
    gamma_q_kernel<<<(n + 63) / 64, 64, 0, ctx->stream>>>(which, n, d, d + n, d + 2 * (size_t)n);
    ctx->launches += 1;
    st = check_cuda(ctx, cudaGetLastError(), "gamma_q_kernel");
  }
  if (st == DPHY_OK) st = check_cuda(ctx, cudaMemcpyAsync(out, d + 2 * (size_t)n, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream), "D2H");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "gamma_q");
  ctx->arena.release(mark);
  return st;
}

int dphy_gamma_q(dphy_ctx* ctx, int32_t n, const double* a, const double* x, double* out) { return gamma_q_call(ctx, 0, n, a, x, out); }
int dphy_gamma_q_inv(dphy_ctx* ctx, int32_t n, const double* a, const double* q, double* out) { return gamma_q_call(ctx, 1, n, a, q, out); }

}  // extern "C"
