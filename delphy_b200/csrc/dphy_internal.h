// dphy_internal.h -- internal structures shared by the host side and the sm_100a kernels.
#ifndef DPHY_INTERNAL_H_
#define DPHY_INTERNAL_H_

#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>
#include <string>
#include <vector>

#include "delphy_b200.h"

namespace dphy {

constexpr int kMaxPartitions = 4;
constexpr int kTile = 256;          // nodes per CTA tile in the SPR / tally kernels (1 node / thread)
constexpr int kLgThreads = 256;     // log-G kernel: threads per CTA
constexpr int kLgNPT = 2;           // log-G kernel: nodes per thread
constexpr int kLgTile = kLgThreads * kLgNPT;   // log-G kernel: nodes per CTA tile

// ---- device arena: the device analogue of the reference's thread-local bump arena (core/scratch_space.h:49-267).
// One slab per ctx, bump-allocated, reset when a "scope" closes.  All temporaries of a launch sequence come from
// here, so the hot path performs no cudaMalloc/cudaFree.
struct Arena {
  char* base = nullptr;
  size_t capacity = 0;
  size_t offset = 0;
  size_t high_water = 0;
  void* alloc(size_t bytes, size_t align = 256) {
    size_t o = (offset + align - 1) / align * align;
    if (o + bytes > capacity) return nullptr;
    offset = o + bytes;
    if (offset > high_water) high_water = offset;
    return base + o;
  }
  size_t mark() const { return offset; }
  void release(size_t m) { offset = m; }
};

// Per-sites-table device view (reference sequence + Global_evo_model + derived tables).
struct SitesDev {
  int32_t L;
  int32_t P;
  const uint8_t* ref;        // [L]
  const uint8_t* part;       // [L]
  const double* nu;          // [L]
  const double* munu;        // [L]  mu_{beta(l)} * nu_l
  const double2* munu2;      // [L]  (mu nu_l, log(mu nu_l)): one 16-byte gather per mutation on the general log-G path (filled when nu_l varies)
  const double* cumQ;        // [L+1] calc_cum_Q_l_for_sequence
  const int32_t* ref_freq;   // [P*4] state frequencies of the reference sequence per partition
  const int32_t* cref;       // [L+1][P*4] cref[l*4P + b*4+a] = #{l' < l : partition(l') == b, ref[l'] == a}  (structure only; 16-byte aligned)
  double mu[kMaxPartitions];
  double pi[kMaxPartitions * 4];
  double q[kMaxPartitions * 16];     // q_ab
  int32_t nu_uniform;        // 1 if every nu_l == nu_const (no site-rate heterogeneity): munu needs no gather
  int32_t pad;
  double nu_const;
  // 64-entry tables indexed by the packed event code (partition << 4 | x << 2 | y), refreshed by every set_evo:
  double tab_dq[kMaxPartitions * 16];   // q_a(y) - q_a(x)
  double tab_md[kMaxPartitions * 16];   // mu nu_const (q_a(y) - q_a(x))              (uniform nu only)
  double tab_lq[kMaxPartitions * 16];   // log(mu nu_const q_xy), 0 on the diagonal   (uniform nu only)
  double tab_muq[kMaxPartitions * 4];   // mu nu_const q_a(a)                          (uniform nu only)
  double tab_logq[kMaxPartitions * 16]; // log(q_xy), 0 on the diagonal: log(mu nu_l q_xy) = munu2[l].y + tab_logq[code]
};

// Per log-G tile descriptor; the tile kernels load it in 16-byte pieces.
struct alignas(16) CTileDesc {
  int32_t tile_start, n_act, node_base, sites_id;   // written by the host at upload
  int32_t cl0, cl1, pad0, pad1;                     // cl*: the tile's slice of the tree's post-order list (closers)
};

// Per-tree record.
struct TreeDev {
  int32_t node_base;       // first device position of this tree
  int32_t num_nodes;
  int32_t sites_id;
  int32_t first_tile;      // index of the tree's first tile in the global tile list
  int32_t num_tiles;
  int32_t includes_run_root;
  int32_t root_id;         // host node index of the root
  int32_t first_ctile;     // log-G (coarse) tiles of kLgTile nodes
  int32_t num_ctiles;
  int32_t pad;
};

// Flattened forest, device order = per tree DFS pre-order visiting children[1] before children[0]
// (the order in which Spr_study_builder emits regions below a start region, core/spr_study.cpp:103-128).
struct ForestDev {
  int32_t num_trees;
  int32_t num_nodes;       // total over trees
  int32_t num_tiles;
  int32_t num_sites_tables;
  int32_t num_ctiles;
  int32_t pad0;
  const TreeDev* trees;
  const SitesDev* sites;
  const int32_t* tile_tree;     // [num_tiles]
  const CTileDesc* ctiles;      // [num_ctiles]
  // per device position
  const int32_t* node_id;       // host node index (within its tree)
  const int32_t* parent_pos;    // device position of the parent (-1 for a root)
  const int32_t* depth;         // depth below the tree's root
  const int32_t* subtree_size;  // nodes in the subtree rooted here (incl. itself)
  const int32_t* post_node;     // per tree: post-order list of device positions
  double* t;                    // node times (mutable: displace moves)
  const int32_t* mut_off;       // [num_nodes+1] CSR, device order
  const int32_t* mut_site;
  const uint8_t* mut_code;      // partition << 4 | from << 2 | to
  double* mut_t;
  const int32_t* miss_off;      // [num_nodes+1]
  const int2* miss_se;          // (start, end) of each missation interval
  const int32_t* fs_off;        // [num_nodes+1]
  const int32_t* fs_site;
  const uint8_t* fs_code;       // partition << 4 | ref << 2 | from
  // from-state overrides folded per branch: fsw[p * fsw_stride + part*4 + a] = #(overrides whose reference state is a)
  // - #(overrides whose from-state is a).  With uniform site rates the branch's delta-lambda term is a 4-term dot product.
  const int16_t* fsw;
  int32_t fsw_stride, pad1;
  // per-node state counts (structure only, built at upload by fold_branch_weights_kernel + the count scan of kernels_flatten.cu).
  // Every per-branch list is folded into one weight vector
  //   bw[p][part*4 + a] = #(mutations to a) - #(mutations from a) - #(sites going missing whose reference state is a)
  //                       + #(overrides whose reference state is a) - #(overrides whose from-state is a),
  // and C is its root -> q prefix:  C[q * fsw_stride + k] = sum of bw[a][k] over the nodes a on the path from the root to q, both
  // included.  ref_freq + C[q] is the state count vector of the sequence at q, so with uniform site rates
  // lambda_i(q) = lambda_ref + sum_k mu nu q_a(a) C[q][k] (core/phylo_tree_calc.h:121-155 summed down the path), and for the root
  // ref_freq + C is the state count vector of calc_log_root_prior (core/phylo_tree_calc.cpp:467-504).
  const int32_t* C;
  // host-order lookup: device position of (tree, host node id) = pos_of_node[tree.node_base + id]
  const int32_t* pos_of_node;
};

// ---- device-side flattening (kernels_flatten.cu) ----------------------------------------------------------------------
// One EMAT as uploaded: the caller's arrays, HOST node order, copied verbatim into a temporary device block.
struct RawTreeDev {
  const int32_t* parent; const int32_t* child0; const int32_t* child1; const double* t;
  const int32_t* mut_off; const int32_t* mut_site; const uint8_t* mut_from; const uint8_t* mut_to; const double* mut_t;
  const int32_t* miss_off; const int32_t* miss_start; const int32_t* miss_end;
  const int32_t* fs_off; const int32_t* fs_site; const uint8_t* fs_from;
  int32_t root, num_nodes, num_muts, num_ivls, num_fs, pad;
};

enum : uint32_t {
  kFlattenErrTopology = 1u,    // not a binary tree rooted at `root` (child/parent mismatch, cycle, unreachable nodes)
  kFlattenErrOffsets = 2u,     // CSR offsets not monotone / inconsistent with the array lengths
  kFlattenErrMutSite = 4u,     // mutation site out of range            (std::out_of_range in the reference)
  kFlattenErrMutState = 8u,    // mutation from/to not in ACGT
  kFlattenErrMissation = 16u,  // missation interval / from-state site out of range (core/mutations.h:187-191)
  kFlattenErrFsState = 32u,    // missation from-state not in ACGT
  kFlattenErrTimes = 64u,      // a node is earlier than its parent (the reference's integrity CHECK, core/phylo_tree.cpp:131)
  kFlattenErrFswRange = 128u,  // more than 32,767 from-state overrides of one (partition, state) on one branch: the folded int16 counts would wrap
};

struct FlattenParams {
  int32_t tile_base = 0;       // first tile of a per-tree launch of the list kernels (flatten_events / fold_branch_weights)
  const TreeDev* trees; const SitesDev* sites; const int32_t* tile_tree; const RawTreeDev* raw;
  int4* arcs[2];               // ping-pong Euler-tour arcs: (succ, #enter arcs to the end, #arcs to the end, -)
  int32_t* scan_tiles;         // [ceil(num_nodes / 1024) * 3]
  uint32_t* status;            // [0] error bits, [1] number of straddlers, then max_depth
  CTileDesc* ctiles; int32_t num_ctiles;
  int32_t* strad_list;         // (device position, sites table) of the nodes whose subtree closes in a later log-G tile than it opens
  int32_t* max_depth;          // [num_trees]
  int32_t num_nodes, total_muts, total_ivls, total_fs;
  // outputs (device order): the ForestDev arrays, writable
  int32_t* node_id; int32_t* parent_pos; int32_t* depth; int32_t* subtree_size; int32_t* post_node; int32_t* pos_of_node;
  double* t;
  int32_t* mut_off; int32_t* mut_site; uint8_t* mut_code; double* mut_t;
  int32_t* miss_off; int2* miss_se;
  int32_t* fs_off; int32_t* fs_site; uint8_t* fs_code;
  int16_t* fsw; int32_t fsw_stride;
  int32_t* C;
  int32_t* cnt_y;              // [num_nodes][fsw_stride] workspace of the count scan: prefix of bw over the post-order lists
  uint4* cnt_tot;              // [ceil(num_nodes / 1024)][fsw_stride / 4][2] its per-tile totals
  // re-flatten of trees whose links did not change (dphy_forest_apply_rows): the DFS order of the forest being replaced is reused
  // and the Euler-tour ranking skipped (null: rank from scratch)
  const int32_t* old_pos_of_node = nullptr; const int32_t* old_depth = nullptr; const int32_t* old_subtree_size = nullptr;
  const int32_t* old_parent_pos = nullptr;
};

// Per-tree index of dphy_forest_place_samples (kernels_place.cu), built by the first placement on the tree.
struct PlaceIndex {
  int32_t R = 0, P2 = 0, L = 0, pad = 0;   // regions of the unbounded study from the root; leaves of the segment tree (power of 2)
  int32_t* site_off = nullptr;             // [L + 1] first record of every site
  int4* rec = nullptr;                     // [M] per mutation, by site: (first region below it, end of those regions, from << 2 | to, dref)
  int2* seg = nullptr;                     // [2 P2] (min, count) segment tree over Hr, leaves at P2 + region
  std::vector<int32_t> h_site_off;         // host copy of site_off (scratch bounds per sample)
  // dated part (dphy_forest_place_dated_samples): a merge-sort tree over region index, keyed by the regions' t_min.  Built by the
  // first dated call that drops a region; it depends on the node and mutation times, so it is rebuilt (in the same block) once
  // dphy_forest_set_node_times has bumped the tree's times version.
  int32_t lg = 0;                          // log2 P2: levels s = 1..lg of the merge-sort tree (level 0 is the segment tree's leaves)
  double* tkey = nullptr;                  // [R] the regions' t_min, ascending (stable: ties by region index); null until first built
  int32_t* lc = nullptr;                   // [lg][P2] level s, entry i of node [a, a + 2^s): how many of its first i - a + 1 entries
                                           // (in t_min order) come from its left child
  int2* pre = nullptr;                     // [lg][P2] level s, entry i: (min Hr, count) over the node's first i - a + 1 entries
  uint64_t dated_at = ~0ull;               // times version the dated part was built at (~0: not valid)
  uint64_t max_at = ~0ull;                 // times version max_key was computed at (~0: not known)
  double max_key = 0.0;                    // the largest t_min: a t_X above it drops no region
};

// One distinct clade of a dphy_clade_table (kernels_clade.cu): its 128-bit key (two wrapping u64 sums of per-tip keys, lanes j = 0
// and 1) and what the trees added so far say about it.  Tables keep keys and values in two arrays sorted by (k0, k1), 32 B a clade.
struct alignas(16) CladeKey { uint64_t k0, k1; };
struct alignas(16) CladeVal { int64_t count; double t_sum; };

}  // namespace dphy

struct dphy_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  dphy::Arena arena;
  std::string last_error;
  int64_t launches = 0;
  void* pinned = nullptr;       // pinned staging buffer for host->device uploads
  size_t pinned_bytes = 0;
  cudaEvent_t pinned_ev = nullptr;   // recorded after the last async copy out of `pinned`
  bool pinned_in_flight = false;
  // second stream for direct (pinned-source) uploads: the list arrays are still in flight over PCIe while the main stream
  // already ranks the Euler tour of the topology arrays that arrived first
  static constexpr int kCopyStreams = 2;   // consecutive DMAs alternate over these, hiding each other's set-up latency (4 measured no better)
  cudaStream_t copy_stream = nullptr;       // == copy_streams[0]: the one the group events are recorded on
  cudaStream_t copy_streams[kCopyStreams] = {};
  cudaEvent_t ev_copy[kCopyStreams] = {};
  std::vector<cudaEvent_t> ev_tree;   // per-tree "lists have landed" events of a direct upload (grown on demand)
  cudaEvent_t ev_main = nullptr, ev_topo = nullptr, ev_nodes = nullptr, ev_lists = nullptr;
  // side stream of the SPR batches: the study-independent template / keep-mask kernels run next to the latency-bound path / X-table
  // chain of the main stream (fork after spr_init_kernel, join before the prefix kernel)
  cudaStream_t aux_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  // tail stream of the SPR batches: the normalisation pass of a batch (bandwidth-bound, touches only the batch's own block) runs
  // here, next to the latency-bound setup chain of the NEXT batch on the main stream; every accessor of the batch joins first
  cudaStream_t tail_stream = nullptr;
  cudaEvent_t ev_tail = nullptr;
  bool tail_dirty = false;      // work has been put on tail_stream since the main stream last joined it
  // Blocks of destroyed SPR batches whose tail may still be running: kept here with the tail's event instead of being returned to
  // the stream-ordered pool (a free in the tail stream's order makes the pool grow by one block per batch while the host enqueues
  // ahead of the device; a free in the main stream's order would make the next batch's set-up wait for the tail).  The next batch
  // takes the OLDEST block -- two batches back, its tail long finished -- after a device-side wait on that event.
  struct SprBlock { void* ptr; size_t bytes; cudaEvent_t ev; };
  std::vector<SprBlock> spr_blocks;
  static constexpr size_t kSprBlocksKept = 3;
  // side streams of the per-site tallies of a whole forest: the trees' (small) kernel sequences run side by side
  static constexpr int kTallyStreams = 4;
  cudaStream_t tally_streams[kTallyStreams] = {};
  cudaEvent_t ev_tally[kTallyStreams] = {};
  struct DeferredCopy { void* dst; const void* src; size_t bytes; };
  std::vector<DeferredCopy> deferred_d2h;   // device->host copies of a batched getter, issued once all its kernels are enqueued
  int logg_path = 0;            // DPHY_LOG_G_PATH_*: 0 auto (folded fast path when every site table has uniform nu), 1 general
};

struct dphy_sites {
  dphy::SitesDev h{};           // host mirror of the device view (pointers are device pointers)
  int32_t L = 0, P = 0;
  uint8_t* d_ref = nullptr; uint8_t* d_part = nullptr; double* d_nu = nullptr; double* d_munu = nullptr; double2* d_munu2 = nullptr;
  double* d_cumQ = nullptr; int32_t* d_ref_freq = nullptr;
  // per-(partition,state) cumulative nu tables for O(1) interval tallies (Ttwiddle): [P*4][L+1]
  double* d_cum_nu_ba = nullptr;
  int32_t* d_cref = nullptr;    // [P*4][L+1] cumulative reference-state counts (structure only; built once at upload)
  size_t bytes = 0;
  uint64_t version = 1;         // bumped by set_evo; forests re-sync their SitesDev copies lazily
};

struct dphy_forest {
  dphy::ForestDev h{};          // host mirror (device pointers)
  std::vector<dphy::TreeDev> trees;
  std::vector<dphy_sites*> sites;
  std::vector<void*> allocs;    // every cudaMalloc'ed block, freed on destroy
  size_t bytes = 0;
  int64_t total_muts = 0, total_ivls = 0, total_fs = 0;
  std::vector<int64_t> tree_muts;     // mutations per tree (incl. the root's list)
  std::vector<int64_t> tree_fs;       // from-state overrides per tree
  std::vector<int32_t> tree_max_depth;
  // host-order arrays of every tree, resident on the device (what dphy_forest_apply_rows patches and re-flattens from)
  std::vector<dphy::RawTreeDev> raw;
  std::vector<int32_t> sites_index;
  // per-node list lengths in host order, mirrored on the host the first time rows are applied: [tree] -> {mut, miss, fs} counts
  std::vector<std::vector<int32_t>> cnt_mut, cnt_miss, cnt_fs;
  // outputs of the last eval (device)
  double* d_lambda = nullptr;   // [num_nodes] device order
  int32_t* d_nsmn = nullptr;    // [num_nodes]
  double* d_tree_out = nullptr; // [num_trees * 4]: root_prior, below_root, T, unused
  int32_t* d_tree_iout = nullptr; // [num_trees * 20]: num_muts, pad, num_muts_ab[16], ...
  // straddlers (log-G): nodes whose subtree crosses a log-G tile boundary; their deltas are precomputed per evaluation
  int32_t* d_strad_list = nullptr; int32_t num_strad = 0;
  double* d_sd_delta = nullptr; int32_t* d_sd_n = nullptr;
  // look-back workspace
  double* d_tile_agg = nullptr;     // [num_tiles]
  int32_t* d_tile_iagg = nullptr;   // [num_tiles]
  uint32_t* d_tile_flag = nullptr;  // [num_tiles]
  double* d_tile_part = nullptr;    // [num_tiles * 2] per-tile partial sums (log G, T)
  int32_t* d_tile_ipart = nullptr;  // [num_tiles * 17]
  const int32_t* d_ctile_order = nullptr;   // [num_ctiles] launch order of the general log-G tile kernel (full tiles first)
  // study-independent tables of the event-scan SPR path (kernels_spr_group2.cuh), built by the first grouped batch on this forest
  int32_t* d_spr_eopen = nullptr; int32_t* d_spr_tnode = nullptr; int32_t* d_spr_ev = nullptr;
  std::vector<dphy::PlaceIndex> place;   // per tree: the placement index (kernels_place.cu), empty until the first placement
  // per tree: bumped by every dphy_forest_set_node_times that gets past argument checks (empty: all 0); the dated placement index
  // compares it with the version it was built at
  std::vector<uint64_t> times_version;
  uint64_t tree_times_version(int tree) const { return (size_t)tree < times_version.size() ? times_version[tree] : 0; }
  bool evaluated = false;
  bool struct_valid = false;    // nsmn / num_muts tallies (structure-only outputs of the general log-G pass) are current
  uint32_t epoch = 0;           // look-back flag value of the current launch (flag == epoch means "published")
  std::vector<uint64_t> sites_version;
  std::vector<uint64_t> eval_version;   // sites versions the last log-G evaluation used (a set_evo since then => stale)
  bool eval_current() const {
    if (!evaluated || eval_version.size() != sites.size()) return false;
    for (size_t i = 0; i < sites.size(); ++i) if (eval_version[i] != sites[i]->version) return false;
    return true;
  }
};

// Clade counts over every tree added so far (kernels_clade.cu).  No pointer to a forest is kept: forests may change or go after an add.
struct dphy_clade_table {
  dphy_ctx* ctx = nullptr;          // the ctx that made the table (its stream orders every use)
  int32_t num_nodes = -1;           // N of every tree, fixed by the first add (-1: nothing added yet)
  int32_t num_tips = 0;             // (N + 1) / 2 for binary trees
  int64_t num_trees = 0;
  int64_t num_clades = 0;
  uint32_t* d_tips = nullptr;       // [(N + 31) / 32] bitmap of the tips' host node indices
  dphy::CladeKey* d_keys = nullptr; // [num_clades] ascending by (k0, k1), unique
  dphy::CladeVal* d_vals = nullptr; // [num_clades] (count, sum of the clade's node time), in d_keys's block
  size_t bytes = 0;                 // resident bytes (bitmap + keys + values)
};

namespace dphy {
// List totals of one tree whose arrays are NOT host-readable (device-resident sources of dphy_forest_apply_rows).
struct TreeTotals { int64_t m, iv, fs, root_m; };
int forest_from_device_arrays(dphy_ctx* ctx, int32_t num_trees, const dphy_emat_host* views, const TreeTotals* totals, const int32_t* sites_index,
                              int32_t num_sites_tables, dphy_sites* const* sites, dphy_forest** out);   // c_abi.cu
int rebuild_forest_from_device(dphy_ctx* ctx, dphy_forest* fo, const dphy_emat_host* trees, const TreeTotals* totals, bool same_links);   // c_abi.cu
int launch_raw_set_node_times(dphy_ctx* ctx, dphy_forest* fo, int tree, const int32_t* d_nodes, const double* d_vals, int count);   // kernels_delta.cu
int set_error(dphy_ctx* ctx, int status, const std::string& msg);
int check_cuda(dphy_ctx* ctx, cudaError_t e, const char* what);
#define DPHY_CUDA(ctx, expr) do { int st__ = dphy::check_cuda((ctx), (expr), #expr); if (st__ != DPHY_OK) return st__; } while (0)

// kernels_sites.cu
int launch_sites_derive(dphy_ctx* ctx, dphy_sites* s, bool with_nu_tables = true);
int launch_sites_ref_counts(dphy_ctx* ctx, dphy_sites* s);
int launch_sites_derive_many(dphy_ctx* ctx, dphy_sites* const* tables, int n);
// kernels_logg.cu
int launch_log_G(dphy_ctx* ctx, dphy_forest* f);            // picks the path (ctx->logg_path, site tables, struct_valid)
int launch_log_G_general(dphy_ctx* ctx, dphy_forest* f);    // every output incl. nsmn and the num_muts tallies
int gather_lambda_host_order(dphy_ctx* ctx, dphy_forest* fo, int tree, double* d_dst);
int gather_nsmn_host_order(dphy_ctx* ctx, dphy_forest* fo, int tree, int32_t* d_dst);
int refresh_sites(dphy_ctx* ctx, dphy_forest* f);   // c_abi.cu
// kernels_flatten.cu
// stage 0: Euler-tour ranking (needs parent / child0 / child1 only); stage 1: node records + CSR offset scans (needs t and the
// three offset arrays); stage 2: list gathers, weight fold, tile descriptors (needs the lists); -1: all
int launch_flatten(dphy_ctx* ctx, const FlattenParams& P, int num_tiles, int max_tree_nodes, int stage = -1);
// stage 2 split per tree (direct uploads: each tree's lists are gathered as soon as its own arrays have landed) ...
int launch_flatten_lists(dphy_ctx* ctx, FlattenParams P, int first_tile, int num_tiles);
// ... then, once every tree's lists are folded: per-node state counts (ForestDev::C), log-G tile descriptors.  launch_flatten
// calls it itself.
int launch_flatten_finish(dphy_ctx* ctx, const FlattenParams& P);
// exclusive scan of n int32 in place (api_tree.cu); tile_tot holds (n + 8191) / 8192 ints
int launch_scan_i32(dphy_ctx* ctx, int32_t* v, int n, int32_t* tile_tot);
// many device-to-device array copies in one launch (16-byte aligned sources and destinations)
struct DeviceCopyJob { char* dst; const char* src; size_t bytes; };
int launch_device_copies(dphy_ctx* ctx, const DeviceCopyJob* d_jobs, int num_jobs, size_t max_bytes);
int launch_set_node_times(dphy_ctx* ctx, dphy_forest* fo, int tree, const int32_t* d_nodes, const double* d_vals, int count, uint32_t* d_status);
// Pinned staging buffer of the ctx: acquire waits for the previous async copy out of it; release records an event.
int acquire_pinned(dphy_ctx* ctx, size_t bytes, void** out);
void release_pinned_async(dphy_ctx* ctx);

// ---- host-side helpers of the entry points ------------------------------------------------------------------------------
constexpr size_t kAlign = 256;
inline size_t align_up(size_t x) { return (x + kAlign - 1) / kAlign * kAlign; }

// A layout planner: reserve() all blocks, then carve them out of one host staging slab and one device slab.
struct Slab {
  struct Block { size_t off, bytes; };
  std::vector<Block> blocks;
  size_t total = 0;
  int reserve(size_t bytes) {
    blocks.push_back({total, bytes});
    total = align_up(total + std::max<size_t>(bytes, 1));
    return (int)blocks.size() - 1;
  }
  template <typename T> T* at(void* base, int id) const { return reinterpret_cast<T*>(static_cast<char*>(base) + blocks[id].off); }
};

// A stream-ordered device allocation, freed when it goes out of scope unless released.
struct DevBlock {
  cudaStream_t s;
  char* p = nullptr;
  explicit DevBlock(cudaStream_t st) : s(st) {}
  DevBlock(DevBlock&& o) noexcept : s(o.s), p(o.release()) {}     // move-only (so that it can live in a std::vector)
  ~DevBlock() { reset(); }
  bool alloc(size_t bytes, cudaError_t* why = nullptr) {
    const cudaError_t e = cudaMallocAsync((void**)&p, std::max<size_t>(bytes, 1), s);
    if (why) *why = e;
    if (e == cudaSuccess) return true;
    p = nullptr;
    cudaGetLastError();
    return false;
  }
  void reset() { if (p) cudaFreeAsync(p, s); p = nullptr; }
  char* release() { char* q = p; p = nullptr; return q; }
};

// The ctx's pinned staging buffer for one call: acquired on construction (check `status`), released once -- by reset() or on
// scope exit -- after the copies out of it have been enqueued.
struct PinnedStage {
  dphy_ctx* ctx;
  char* p = nullptr;
  int status; bool held;
  PinnedStage(dphy_ctx* c, size_t bytes) : ctx(c) {
    void* v = nullptr;
    status = acquire_pinned(c, bytes, &v);
    held = status == DPHY_OK;
    p = static_cast<char*>(v);
  }
  PinnedStage(PinnedStage&&) = delete;
  ~PinnedStage() { reset(); }
  void reset() { if (held) release_pinned_async(ctx); held = false; }
};

// bits of a radix-sort key that holds 0 .. max_value (at least 1, at most 31)
inline int bits_for(int64_t max_value) { int b = 1; while (b < 31 && ((int64_t)1 << b) <= max_value) ++b; return b; }
}  // namespace dphy

#endif  // DPHY_INTERNAL_H_
