// kernels_delta.cu -- device-resident incremental EMAT updates (SURVEY.md section 8f row 1).
//
// The reference edits its Phylo_tree in place between hot-path calls: an accepted branch-reform move rewrites one branch's
// mutation list (core/subrun.cpp:316-319, core/phylo_tree.cpp:579-644); an SPR move (Spr_move::peel_graft / move / apply_graft,
// core/spr_move.cpp:838-1156, through Tree_editing_session, core/tree_editing.cpp) touches the O(path) nodes around P: their
// parent / children links, times, mutation lists, missation intervals and from-states, possibly the root.  dphy_forest_apply_rows
// mirrors such edits on the device: the caller sends only the rows (nodes) that changed; the host-order arrays of every tree stay
// resident next to the flattened forest, the changed trees' arrays are rebuilt on the device (new CSR offsets by a scan of the
// patched list lengths, lists gathered from the old arrays or from the uploaded rows), and the forest is re-flattened from
// there by the same kernels as an upload -- nothing but the changed rows crosses PCIe, and the host never re-walks the tree.
#include "dphy_internal.h"
#include "device_utils.cuh"

#include <algorithm>
#include <cstring>
#include <vector>

namespace dphy {

// one changed node, device form; list payloads live in one packed buffer at the given element offsets
struct RowDev {
  int32_t node, parent, child0, child1;
  double t;
  int32_t n_muts, n_miss, n_fs, pad;
  int32_t o_mut, o_miss, o_fs, pad2;    // element offsets into the payload arrays
};

struct RowPayloadDev {
  const RowDev* rows;
  const int32_t* mut_site; const uint8_t* mut_from; const uint8_t* mut_to; const double* mut_t;
  const int32_t* miss_start; const int32_t* miss_end;
  const int32_t* fs_site; const uint8_t* fs_from;
};

struct RawTreeOut {     // writable twin of RawTreeDev
  int32_t* parent; int32_t* child0; int32_t* child1; double* t;
  int32_t* mut_off; int32_t* mut_site; uint8_t* mut_from; uint8_t* mut_to; double* mut_t;
  int32_t* miss_off; int32_t* miss_start; int32_t* miss_end;
  int32_t* fs_off; int32_t* fs_site; uint8_t* fs_from;
};

// row_of[v] = index of the row that replaces node v, or -1
__global__ void delta_mark_kernel(int32_t* __restrict__ row_of, int num_nodes, const RowDev* __restrict__ rows, int row0, int row1) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < num_nodes) row_of[i] = -1;
}
__global__ void delta_mark_rows_kernel(int32_t* __restrict__ row_of, const RowDev* __restrict__ rows, int row0, int row1, RawTreeDev old,
                                       uint32_t* __restrict__ links_changed) {
  const int i = row0 + blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= row1) return;
  const RowDev r = rows[i];
  row_of[r.node] = i;      // a node listed twice: the later row wins deterministically only if callers avoid it (checked on the host)
  // a row that keeps its node's links (displacements, branch reforms) leaves the DFS order alone: the re-flatten then skips the ranking
  if (r.parent != old.parent[r.node] || r.child0 != old.child0[r.node] || r.child1 != old.child1[r.node]) atomicOr(links_changed, 1u);
}

// New CSR offsets of the three lists (blockIdx.y = list kind) from the patched per-node lengths, two levels: every CTA scans one
// tile of 8,192 nodes (tile-local exclusive prefix + the tile total), then every tile adds the totals of the tiles before it.
// (One CTA per list walking the whole tree with a running carry took 277 us per 100k-tip tree: 196 rounds of dependent gathers.)
constexpr int kDeltaTile = 1024 * 8;
__global__ void __launch_bounds__(1024) delta_offsets_kernel(RawTreeDev old, RawTreeOut out, const int32_t* __restrict__ row_of,
                                                             const RowDev* __restrict__ rows, int32_t* __restrict__ tile_tot) {
  __shared__ int s_ws[32];
  const int kind = blockIdx.y;
  const int32_t* old_off = kind == 0 ? old.mut_off : (kind == 1 ? old.miss_off : old.fs_off);
  int32_t* new_off = kind == 0 ? out.mut_off : (kind == 1 ? out.miss_off : out.fs_off);
  const int n = old.num_nodes;
  const int v0 = blockIdx.x * kDeltaTile;
  int cnt[8], mine = 0;
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const int v = v0 + (int)threadIdx.x * 8 + u;
    cnt[u] = 0;
    if (v < n) {
      const int r = row_of[v];
      cnt[u] = r < 0 ? old_off[v + 1] - old_off[v] : (kind == 0 ? rows[r].n_muts : (kind == 1 ? rows[r].n_miss : rows[r].n_fs));
    }
    mine += cnt[u];
  }
  int tot;
  const int incl = block_scan_incl<int, 1024>(mine, s_ws, &tot);
  int run = incl - mine;
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const int v = v0 + (int)threadIdx.x * 8 + u;
    if (v < n) new_off[v] = run;
    run += cnt[u];
  }
  if (threadIdx.x == 0) tile_tot[kind * gridDim.x + blockIdx.x] = tot;
}
__global__ void __launch_bounds__(1024) delta_offsets_fix_kernel(RawTreeOut out, int n, const int32_t* __restrict__ tile_tot) {
  const int kind = blockIdx.y;
  int32_t* new_off = kind == 0 ? out.mut_off : (kind == 1 ? out.miss_off : out.fs_off);
  const int32_t* tt = tile_tot + kind * gridDim.x;
  int base = 0;
  for (int t = 0; t < (int)blockIdx.x; ++t) base += __ldg(tt + t);
  const int v0 = blockIdx.x * kDeltaTile;
  if (base) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int v = v0 + u * 1024 + (int)threadIdx.x;
      if (v < n) new_off[v] += base;
    }
  }
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) new_off[n] = base + __ldg(tt + blockIdx.x);
}

// One thread per node: node scalars + its three lists, from the row that replaces it or from the old arrays.
__global__ void delta_gather_kernel(RawTreeDev old, RawTreeOut out, const int32_t* __restrict__ row_of, RowPayloadDev P) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= old.num_nodes) return;
  const int r = row_of[v];
  int mo = out.mut_off[v], io = out.miss_off[v], fo = out.fs_off[v];
  if (r < 0) {
    out.parent[v] = old.parent[v]; out.child0[v] = old.child0[v]; out.child1[v] = old.child1[v]; out.t[v] = old.t[v];
    for (int i = old.mut_off[v]; i < old.mut_off[v + 1]; ++i, ++mo) {
      out.mut_site[mo] = old.mut_site[i]; out.mut_from[mo] = old.mut_from[i]; out.mut_to[mo] = old.mut_to[i]; out.mut_t[mo] = old.mut_t[i];
    }
    for (int i = old.miss_off[v]; i < old.miss_off[v + 1]; ++i, ++io) { out.miss_start[io] = old.miss_start[i]; out.miss_end[io] = old.miss_end[i]; }
    for (int i = old.fs_off[v]; i < old.fs_off[v + 1]; ++i, ++fo) { out.fs_site[fo] = old.fs_site[i]; out.fs_from[fo] = old.fs_from[i]; }
  } else {
    const RowDev R = P.rows[r];
    out.parent[v] = R.parent; out.child0[v] = R.child0; out.child1[v] = R.child1; out.t[v] = R.t;
    for (int i = 0; i < R.n_muts; ++i, ++mo) {
      out.mut_site[mo] = P.mut_site[R.o_mut + i]; out.mut_from[mo] = P.mut_from[R.o_mut + i]; out.mut_to[mo] = P.mut_to[R.o_mut + i];
      out.mut_t[mo] = P.mut_t[R.o_mut + i];
    }
    for (int i = 0; i < R.n_miss; ++i, ++io) { out.miss_start[io] = P.miss_start[R.o_miss + i]; out.miss_end[io] = P.miss_end[R.o_miss + i]; }
    for (int i = 0; i < R.n_fs; ++i, ++fo) { out.fs_site[fo] = P.fs_site[R.o_fs + i]; out.fs_from[fo] = P.fs_from[R.o_fs + i]; }
  }
}

// the raw copy of the node times follows dphy_forest_set_node_times, so that a later apply_rows starts from the current times
__global__ void raw_set_node_times_kernel(double* __restrict__ raw_t, int num_nodes, const int32_t* __restrict__ nodes,
                                          const double* __restrict__ vals, int count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const int v = nodes[i];
  if (v >= 0 && v < num_nodes) raw_t[v] = vals[i];
}

int launch_raw_set_node_times(dphy_ctx* ctx, dphy_forest* fo, int tree, const int32_t* d_nodes, const double* d_vals, int count) {
  if (tree < 0 || tree >= (int)fo->raw.size() || count <= 0) return DPHY_OK;
  raw_set_node_times_kernel<<<(count + 255) / 256, 256, 0, ctx->stream>>>(const_cast<double*>(fo->raw[tree].t), fo->raw[tree].num_nodes, d_nodes, d_vals, count);
  ctx->launches += 1;
  return check_cuda(ctx, cudaGetLastError(), "raw_set_node_times_kernel");
}

}  // namespace dphy

using namespace dphy;

namespace {
// per-node list lengths, host order, fetched once from the resident raw offsets
int ensure_host_counts(dphy_ctx* ctx, dphy_forest* fo) {
  const int nt = fo->h.num_trees;
  if ((int)fo->cnt_mut.size() == nt) return DPHY_OK;
  fo->cnt_mut.assign(nt, {}); fo->cnt_miss.assign(nt, {}); fo->cnt_fs.assign(nt, {});
  std::vector<int32_t> off;
  for (int k = 0; k < nt; ++k) {
    const RawTreeDev& R = fo->raw[k];
    const int n = R.num_nodes;
    const int32_t* srcs[3] = {R.mut_off, R.miss_off, R.fs_off};
    std::vector<int32_t>* dsts[3] = {&fo->cnt_mut[k], &fo->cnt_miss[k], &fo->cnt_fs[k]};
    for (int j = 0; j < 3; ++j) {
      off.resize(n + 1);
      DPHY_CUDA(ctx, cudaMemcpyAsync(off.data(), srcs[j], sizeof(int32_t) * (n + 1), cudaMemcpyDeviceToHost, ctx->stream));
      DPHY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
      dsts[j]->resize(n);
      for (int v = 0; v < n; ++v) (*dsts[j])[v] = off[v + 1] - off[v];
    }
  }
  return DPHY_OK;
}
}  // namespace

extern "C" int dphy_forest_apply_rows(dphy_ctx* ctx, dphy_forest* fo, int32_t count, const dphy_node_row* rows, const int32_t* new_roots) {
  if (!ctx || !fo || count < 0 || (count > 0 && !rows)) return DPHY_ERR_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  const int nt = fo->h.num_trees;
  if ((int)fo->raw.size() != nt) return set_error(ctx, DPHY_ERR_INTERNAL, "apply_rows: the forest holds no resident raw arrays");
  int st = ensure_host_counts(ctx, fo);
  if (st != DPHY_OK) return st;

  // ---- validate, group by tree, size the payload ------------------------------------------------------------------------------------------
  std::vector<std::vector<int>> by_tree(nt);
  size_t pm = 0, pi = 0, pf = 0;
  for (int i = 0; i < count; ++i) {
    const dphy_node_row& r = rows[i];
    if (r.tree < 0 || r.tree >= nt) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "apply_rows: tree index out of range");
    const int n = fo->raw[r.tree].num_nodes;
    if (r.node < 0 || r.node >= n) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "apply_rows: node out of range");
    if (r.parent < -1 || r.parent >= n || r.child0 < -1 || r.child0 >= n || r.child1 < -1 || r.child1 >= n)
      return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "apply_rows: parent / child index out of range");
    if (r.n_muts < 0 || r.n_miss < 0 || r.n_fs < 0) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "apply_rows: negative list length");
    if ((r.n_muts > 0 && (!r.mut_site || !r.mut_from || !r.mut_to || !r.mut_t)) || (r.n_miss > 0 && (!r.miss_start || !r.miss_end)) ||
        (r.n_fs > 0 && (!r.fs_site || !r.fs_from)))
      return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "apply_rows: a list length without its arrays");
    for (int j : by_tree[r.tree]) if (rows[j].node == r.node) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "apply_rows: a node is listed twice");
    by_tree[r.tree].push_back(i);
    pm += r.n_muts; pi += r.n_miss; pf += r.n_fs;
  }
  bool any = false;
  for (int k = 0; k < nt; ++k) any = any || !by_tree[k].empty() || (new_roots && new_roots[k] != fo->raw[k].root);
  if (!any) return DPHY_OK;

  // ---- pack rows + payload into the pinned slab, one H2D ----------------------------------------------------------------------------------
  Slab pay;
  const int b_rows = pay.reserve(sizeof(RowDev) * std::max(1, count)), b_msite = pay.reserve(4 * pm), b_mfrom = pay.reserve(pm);
  const int b_mto = pay.reserve(pm), b_mt = pay.reserve(8 * pm), b_is = pay.reserve(4 * pi), b_ie = pay.reserve(4 * pi);
  const int b_fsite = pay.reserve(4 * pf), b_ffrom = pay.reserve(pf);
  PinnedStage pin(ctx, pay.total);
  if (pin.status != DPHY_OK) return pin.status;
  char* hb = pin.p;
  RowDev* hrows = pay.at<RowDev>(hb, b_rows);
  {
    size_t cm = 0, ci = 0, cf = 0;
    // rows grouped tree-major so that each tree's kernels address one contiguous range
    int w = 0;
    std::vector<int> order; order.reserve(count);
    for (int k = 0; k < nt; ++k) for (int j : by_tree[k]) order.push_back(j);
    for (int j : order) {
      const dphy_node_row& r = rows[j];
      RowDev& d = hrows[w++];
      d.node = r.node; d.parent = r.parent; d.child0 = r.child0; d.child1 = r.child1; d.t = r.t;
      d.n_muts = r.n_muts; d.n_miss = r.n_miss; d.n_fs = r.n_fs; d.pad = 0; d.pad2 = 0;
      d.o_mut = (int32_t)cm; d.o_miss = (int32_t)ci; d.o_fs = (int32_t)cf;
      if (r.n_muts) {
        std::memcpy(pay.at<int32_t>(hb, b_msite) + cm, r.mut_site, 4 * (size_t)r.n_muts); std::memcpy(pay.at<uint8_t>(hb, b_mfrom) + cm, r.mut_from, r.n_muts);
        std::memcpy(pay.at<uint8_t>(hb, b_mto) + cm, r.mut_to, r.n_muts); std::memcpy(pay.at<double>(hb, b_mt) + cm, r.mut_t, 8 * (size_t)r.n_muts);
      }
      if (r.n_miss) { std::memcpy(pay.at<int32_t>(hb, b_is) + ci, r.miss_start, 4 * (size_t)r.n_miss); std::memcpy(pay.at<int32_t>(hb, b_ie) + ci, r.miss_end, 4 * (size_t)r.n_miss); }
      if (r.n_fs) { std::memcpy(pay.at<int32_t>(hb, b_fsite) + cf, r.fs_site, 4 * (size_t)r.n_fs); std::memcpy(pay.at<uint8_t>(hb, b_ffrom) + cf, r.fs_from, r.n_fs); }
      cm += r.n_muts; ci += r.n_miss; cf += r.n_fs;
    }
  }
  // payload, link flag, new raw blocks + row maps: consumed by the re-flatten below, freed stream-ordered after it
  std::vector<DevBlock> scratch;
  scratch.emplace_back(ctx->stream);
  if (!scratch.back().alloc(pay.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(rows)");
  char* d_pay = scratch.back().p;
  cudaError_t ce = cudaMemcpyAsync(d_pay, hb, pay.total, cudaMemcpyHostToDevice, ctx->stream);
  pin.reset();
  if (ce != cudaSuccess) return check_cuda(ctx, ce, "H2D rows");
  RowPayloadDev P{};
  P.rows = pay.at<const RowDev>(d_pay, b_rows);
  P.mut_site = pay.at<const int32_t>(d_pay, b_msite); P.mut_from = pay.at<const uint8_t>(d_pay, b_mfrom);
  P.mut_to = pay.at<const uint8_t>(d_pay, b_mto); P.mut_t = pay.at<const double>(d_pay, b_mt);
  P.miss_start = pay.at<const int32_t>(d_pay, b_is); P.miss_end = pay.at<const int32_t>(d_pay, b_ie);
  P.fs_site = pay.at<const int32_t>(d_pay, b_fsite); P.fs_from = pay.at<const uint8_t>(d_pay, b_ffrom);

  // ---- rebuild the raw arrays of every changed tree on the device ----------------------------------------------------------------------------
  std::vector<dphy_emat_host> views(nt);
  std::vector<TreeTotals> totals(nt);
  // one word: set by a row whose links differ from its node's current ones
  scratch.emplace_back(ctx->stream);
  if (!scratch.back().alloc(256)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(apply_rows flag)");
  uint32_t* d_links = reinterpret_cast<uint32_t*>(scratch.back().p);
  cudaMemsetAsync(d_links, 0, sizeof(uint32_t), ctx->stream);
  bool root_changed = false;
  int row0 = 0;
  struct TreeJob { RawTreeDev R; RawTreeOut out; int32_t* row_of; int32_t* tt; int n, ntiles, row0, nrows; };
  std::vector<TreeJob> jobs;        // the edited trees: blocks allocated first (main stream), kernels launched after the fork below
  for (int k = 0; k < nt; ++k) {
    const RawTreeDev& R = fo->raw[k];
    if (new_roots && new_roots[k] != R.root) root_changed = true;
    const int n = R.num_nodes;
    dphy_emat_host& e = views[k];
    std::memset(&e, 0, sizeof(e));
    e.num_nodes = n; e.root = new_roots ? new_roots[k] : R.root; e.includes_run_root = fo->trees[k].includes_run_root;
    if (e.root < 0 || e.root >= n) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "apply_rows: new root out of range");
    // the host mirror of the list lengths is updated only once the rebuild has succeeded (a node has at most one row per tree)
    int64_t M = R.num_muts, I = R.num_ivls, F = R.num_fs, root_m = fo->cnt_mut[k][e.root];
    for (int j : by_tree[k]) {
      const dphy_node_row& r = rows[j];
      M += r.n_muts - fo->cnt_mut[k][r.node]; I += r.n_miss - fo->cnt_miss[k][r.node]; F += r.n_fs - fo->cnt_fs[k][r.node];
      if (r.node == e.root) root_m = r.n_muts;
    }
    totals[k] = {M, I, F, root_m};
    const int nrows = (int)by_tree[k].size();
    if (nrows == 0) {
      // untouched tree: re-flattened from the arrays it already has
      e.parent = R.parent; e.child0 = R.child0; e.child1 = R.child1; e.t = R.t;
      e.mut_off = R.mut_off; e.mut_site = R.mut_site; e.mut_from = R.mut_from; e.mut_to = R.mut_to; e.mut_t = R.mut_t;
      e.miss_off = R.miss_off; e.miss_start = R.miss_start; e.miss_end = R.miss_end;
      e.fs_off = R.fs_off; e.fs_site = R.fs_site; e.fs_from = R.fs_from;
      continue;
    }
    Slab raw;
    const int a_par = raw.reserve(4 * (size_t)n), a_c0 = raw.reserve(4 * (size_t)n), a_c1 = raw.reserve(4 * (size_t)n), a_t = raw.reserve(8 * (size_t)n);
    const int a_moff = raw.reserve(4 * ((size_t)n + 1)), a_msite = raw.reserve(4 * M), a_mfrom = raw.reserve(M), a_mto = raw.reserve(M), a_mt = raw.reserve(8 * M);
    const int a_ioff = raw.reserve(4 * ((size_t)n + 1)), a_is = raw.reserve(4 * I), a_ie = raw.reserve(4 * I);
    const int a_foff = raw.reserve(4 * ((size_t)n + 1)), a_fsite = raw.reserve(4 * F), a_ffrom = raw.reserve(F), a_map = raw.reserve(4 * (size_t)n);
    const int ntiles = (n + kDeltaTile - 1) / kDeltaTile;
    const int a_tt = raw.reserve(4 * 3 * (size_t)ntiles);
    scratch.emplace_back(ctx->stream);
    if (!scratch.back().alloc(raw.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(raw rebuild)");
    char* nb = scratch.back().p;
    RawTreeOut out{};
    out.parent = raw.at<int32_t>(nb, a_par); out.child0 = raw.at<int32_t>(nb, a_c0); out.child1 = raw.at<int32_t>(nb, a_c1); out.t = raw.at<double>(nb, a_t);
    out.mut_off = raw.at<int32_t>(nb, a_moff); out.mut_site = raw.at<int32_t>(nb, a_msite); out.mut_from = raw.at<uint8_t>(nb, a_mfrom);
    out.mut_to = raw.at<uint8_t>(nb, a_mto); out.mut_t = raw.at<double>(nb, a_mt);
    out.miss_off = raw.at<int32_t>(nb, a_ioff); out.miss_start = raw.at<int32_t>(nb, a_is); out.miss_end = raw.at<int32_t>(nb, a_ie);
    out.fs_off = raw.at<int32_t>(nb, a_foff); out.fs_site = raw.at<int32_t>(nb, a_fsite); out.fs_from = raw.at<uint8_t>(nb, a_ffrom);
    jobs.push_back({R, out, raw.at<int32_t>(nb, a_map), raw.at<int32_t>(nb, a_tt), n, ntiles, row0, nrows});
    row0 += nrows;
    e.parent = out.parent; e.child0 = out.child0; e.child1 = out.child1; e.t = out.t;
    e.mut_off = out.mut_off; e.mut_site = out.mut_site; e.mut_from = out.mut_from; e.mut_to = out.mut_to; e.mut_t = out.mut_t;
    e.miss_off = out.miss_off; e.miss_start = out.miss_start; e.miss_end = out.miss_end;
    e.fs_off = out.fs_off; e.fs_site = out.fs_site; e.fs_from = out.fs_from;
  }
  // Every edited tree's sequence is five small kernels (25 - 800 CTAs each): tree j runs on side stream j % 4, forked after the
  // allocations and the payload upload on the main stream, joined before the re-flatten
  {
    constexpr int kS = dphy_ctx::kTallyStreams;
    cudaStream_t main_stream = ctx->stream;
    bool forked = false;
    if (jobs.size() > 1) {
      bool ok = true;
      for (int i = 0; i < kS && ok; ++i) {
        if (!ctx->tally_streams[i]) ok = cudaStreamCreateWithFlags(&ctx->tally_streams[i], cudaStreamNonBlocking) == cudaSuccess &&
                                         cudaEventCreateWithFlags(&ctx->ev_tally[i], cudaEventDisableTiming) == cudaSuccess;
      }
      if (ok && !ctx->ev_fork) ok = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) == cudaSuccess;
      if (ok) {
        cudaEventRecord(ctx->ev_fork, main_stream);
        for (int i = 0; i < kS; ++i) cudaStreamWaitEvent(ctx->tally_streams[i], ctx->ev_fork, 0);
        forked = true;
      } else cudaGetLastError();
    }
    for (size_t j = 0; j < jobs.size(); ++j) {
      const TreeJob& J = jobs[j];
      cudaStream_t s = forked ? ctx->tally_streams[j % kS] : main_stream;
      delta_mark_kernel<<<(J.n + 255) / 256, 256, 0, s>>>(J.row_of, J.n, P.rows, J.row0, J.row0 + J.nrows);
      delta_mark_rows_kernel<<<(J.nrows + 255) / 256, 256, 0, s>>>(J.row_of, P.rows, J.row0, J.row0 + J.nrows, J.R, d_links);
      delta_offsets_kernel<<<dim3(J.ntiles, 3), 1024, 0, s>>>(J.R, J.out, J.row_of, P.rows, J.tt);
      delta_offsets_fix_kernel<<<dim3(J.ntiles, 3), 1024, 0, s>>>(J.out, J.n, J.tt);
      delta_gather_kernel<<<(J.n + 255) / 256, 256, 0, s>>>(J.R, J.out, J.row_of, P);
      ctx->launches += 5;
    }
    if (forked)
      for (int i = 0; i < kS; ++i) { cudaEventRecord(ctx->ev_tally[i], ctx->tally_streams[i]); cudaStreamWaitEvent(main_stream, ctx->ev_tally[i], 0); }
  }
  st = check_cuda(ctx, cudaGetLastError(), "apply_rows kernels");
  uint32_t links = 1u;
  if (st == DPHY_OK) st = check_cuda(ctx, cudaMemcpyAsync(&links, d_links, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream), "D2H");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "apply_rows");
  const bool same_links = links == 0u && !root_changed;
  // ---- re-flatten from the device-resident arrays (the same kernels as an upload; validation included) ----------------------------------------------
  if (st == DPHY_OK) st = rebuild_forest_from_device(ctx, fo, views.data(), totals.data(), same_links);
  scratch.clear();
  if (st != DPHY_OK) return st;
  for (int k = 0; k < nt; ++k)
    for (int j : by_tree[k]) {
      const dphy_node_row& r = rows[j];
      fo->cnt_mut[k][r.node] = r.n_muts; fo->cnt_miss[k][r.node] = r.n_miss; fo->cnt_fs[k][r.node] = r.n_fs;
    }
  return DPHY_OK;
}
