// kernels_spr_frontier.cuh -- bounded SPR studies (max_muts_from_start small: what Subrun::spr1_move issues 99 % of the time,
// core/subrun.cpp:495-499) as a walk of the ball itself.  (included by kernels_spr.cu inside namespace dphy)
//
// The per-study pipeline sweeps all N nodes of the tree (two scans, the segments, the emit) to produce the few dozen regions of a
// ball of radius 1; here ONE THREAD per study walks exactly the regions the reference's builder visits, in its order, so the work is
// proportional to the ball.  The builder's explicit LIFO work stack (Spr_study_builder::do_pending_work / seed_neighbors_except,
// core/spr_study.cpp:26-41,103-128) is not needed: the regions form a tree, so the walk is a depth-first traversal of that tree
// re-rooted at the start region, and both "where did I come from" and "which neighbour is next" follow from positions alone --
//   * the neighbours of region (p, k), in the order the builder VISITS them (reverse of its pushes): the next region down the branch
//     (p, k+1), or, at the bottom of an inner branch, the top regions of children[1] then children[0] (device positions p + 1 and
//     p + 1 + subtree_size[p + 1]); then the region above: (p, k-1), or the parent's bottom region;
//   * the neighbour that leads back to the start region: for a node that is a proper ancestor of the start node it is the
//     neighbour BELOW (towards the start), on the start branch it is the one towards k0, everywhere else it is the one above.
// Crossing mutation m changes the counted-mutation distance by one (unless its site is missing at X) and the Hamming potential by
// d(m) (kernels_spr.cu header): min_muts(region) = init_min_muts + H(region) - H(start), as in the other pipelines.
// account_for_Xs_detachment (:130-209) and remove_regions_in_Xs_future (:211-224) are then applied to the short list in place.
//
// The walk is a chain of dependent loads, so a study gets a whole warp, not a thread: at every region lanes 0-2 evaluate the three
// neighbours at once (target, the mutation crossed, its count and potential from X's state table) and lane 3 the way back, and on
// arrival at a new node the lanes fetch its attributes side by side; a step costs ~4 load latencies however many neighbours are
// rejected.  Regions that start at or after t_X, and everything below them, are not walked (the builder walks them and drops them
// afterwards).  Measured on a 100k-tip tree, radius 1 (~22 regions per study): 7.0 us per study in a batch of 64, 3.4 in a batch of
// 512 -- the O(N) sweeps of the per-study pipeline: 9.7 / 7.9 (tools/spr_bounded_timing.py; one thread per study: 15.5).
struct FRegion { int p, k; };

__global__ void __launch_bounds__(128) spr_frontier_kernel(ForestDev f, SprBatchDev B) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int study = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (study >= B.num_studies) return;
  SprStudy& S = B.studies[study];
  if (S.h_stride != 0 || S.error) return;              // h_stride 0 marks the studies of this kernel
  const uint8_t* __restrict__ xtab = (const uint8_t*)(B.slab + S.off_xtab);
  RegionHead* out = (RegionHead*)(B.slab + S.off_regions);
  const int p0 = S.pos0, k0 = S.k0, posX = S.posX, root = S.root_pos, limit = S.limit, cap = S.region_cap;
  const int init_mm = S.init_min_muts, posS = S.posS, posP = S.posP;
  const double tX = S.t_X;
  if (lane == 0) S.mu = S.lambda_X / (double)(S.L - S.num_missing);   // Spr_study::mu, core/spr_study.cpp:239 (spr_segments_kernel does it elsewhere)
  int n_out = 0;
  bool overflow = false;

  // ---- attributes of the current node (warp-uniform), fetched side by side -----------------------------------------------------------------
  int p = p0, k = k0, moff = 0, np = 0, size = 1, par = -1, idn = 0, size_c1 = 1, np_par = 0;
  double tN = 0.0, tP = 0.0;
  auto load_node = [&](int q) {
    // level 1: lane i fetches one attribute of q; level 2: what hangs off the parent
    int v = 0; double d = 0.0;
    if (lane == 0) v = f.mut_off[q];
    else if (lane == 1) v = f.mut_off[q + 1];
    else if (lane == 2) v = f.subtree_size[q];
    else if (lane == 3) v = f.parent_pos[q];
    else if (lane == 4) v = f.node_id[q];
    else if (lane == 5) d = f.t[q];
    else if (lane == 6 && q + 1 < f.num_nodes) v = f.subtree_size[q + 1];     // children[1] of an inner node (unused for a leaf)
    moff = __shfl_sync(full, v, 0); np = __shfl_sync(full, v, 1) - moff; size = __shfl_sync(full, v, 2); par = __shfl_sync(full, v, 3);
    idn = __shfl_sync(full, v, 4); tN = __shfl_sync(full, d, 5); size_c1 = __shfl_sync(full, v, 6);
    int w = 0; double e = 0.0;
    if (par >= 0) {
      if (lane == 0) w = f.mut_off[par];
      else if (lane == 1) w = f.mut_off[par + 1];
      else if (lane == 2) e = f.t[par];
    }
    np_par = __shfl_sync(full, w, 1) - __shfl_sync(full, w, 0); tP = __shfl_sync(full, e, 2);
    p = q;
  };
  auto emit = [&](int H) {
    if (n_out >= cap) { overflow = true; return; }
    const bool is_root = p == root;
    double a = 0.0;
    if (lane == 0 && k > 0) a = f.mut_t[moff + k - 1];
    else if (lane == 1 && k < np) a = f.mut_t[moff + k];
    const double mt_prev = __shfl_sync(full, a, 0), mt_next = __shfl_sync(full, a, 1);
    if (lane == 0) {
      RegionHead h;
      h.branch = idn; h.mut_idx = k;
      h.t_min = is_root ? -DBL_MAX : (k == 0 ? tP : mt_prev);        // spr_study.h:90-95
      h.t_max = (is_root || k == np) ? tN : mt_next;                 // spr_study.h:96-101
      h.min_muts = init_mm + H; h.pad = 0;
      out[n_out] = h;
    }
    ++n_out;
  };

  // ---- the walk -------------------------------------------------------------------------------------------------------------------------
  load_node(p0);
  if (size <= 1) size_c1 = 1;
  int C = 0, H = 0, next = 0;
  emit(H);
  for (long long guard = 0; guard < (1LL << 40) && !overflow; ++guard) {
    // the neighbour that leads back to the start region (p = -1 at the start region itself)
    FRegion back; back.p = -1; back.k = 0;
    if (p == p0) { if (k != k0) { back.p = p; back.k = k > k0 ? k - 1 : k + 1; } }
    else if (p < p0 && p0 < p + size) {                 // proper ancestor of the start node: back = down
      if (k < np) { back.p = p; back.k = k + 1; }
      else { const int c1 = p + 1; back.p = (p0 < c1 + size_c1) ? c1 : c1 + size_c1; back.k = 0; }
    } else if (par >= 0) {
      if (k > 0) { back.p = p; back.k = k - 1; } else { back.p = par; back.k = np_par; }
    }
    // lanes 0-2: neighbour number `lane` in visiting order; lane 3: the way back.  Each with the mutation it crosses, if any.
    FRegion n; n.p = -1; n.k = 0;
    if (lane == 0) { if (k < np) { n.p = p; n.k = k + 1; } else if (size > 1) { n.p = p + 1; } }
    else if (lane == 1) { if (k == np && size > 1) n.p = p + 1 + size_c1; }
    else if (lane == 2) { if (par >= 0) { if (k > 0) { n.p = p; n.k = k - 1; } else { n.p = par; n.k = np_par; } } }
    else if (lane == 3) n = back;
    int dC = 0, dH = 0;
    bool future = false;
    if (lane < 4 && n.p == p) {                         // same branch: one mutation crossed
      const int i = moff + min(k, n.k);
      const int xt = xtab[f.mut_site[i]];
      if (!(xt & 4)) { dC = 1; const int d = g_mut_dh(xt, f.mut_code[i] & 15); dH = n.k > k ? d : -d; }
      // Everything below a region that starts at or after t_X starts after t_X too and is dropped by remove_regions_in_Xs_future:
      // the builder walks it all the same (mutation-free clades make the radius-1 ball heavy-tailed), we do not.  S and P are
      // exempt: account_for_Xs_detachment moves the start of their regions.
      if (lane == 0 && p != posS && p != posP) future = f.mut_t[i] >= tX;
    } else if (lane < 2 && n.p >= 0 && n.p != posS && n.p != posP) {
      future = tN >= tX;                                // top region of a child: starts at this node's time
    }
    const bool fwd = lane < 3 && lane >= next && n.p >= 0 && !(n.p == back.p && n.k == back.k) && !future &&
                     n.p != posX && C + dC <= limit;     // Spr_study_builder::is_cur_region_in_scope, core/spr_study.h:86-89
    const unsigned go = __ballot_sync(full, fwd);
    if (go) {
      const int src = __ffs(go) - 1;
      const int q = __shfl_sync(full, n.p, src), kk = __shfl_sync(full, n.k, src);
      C += __shfl_sync(full, dC, src); H += __shfl_sync(full, dH, src);
      if (q != p) { load_node(q); if (size <= 1) size_c1 = 1; }
      k = kk; next = 0;
      emit(H);
    } else {
      // every neighbour done or out of scope: step back towards the start region, undoing the crossing, and resume after this
      // region in the neighbour list of the one we return to
      if (back.p < 0) break;
      C -= __shfl_sync(full, dC, 3); H += __shfl_sync(full, dH, 3);
      int idx;
      if (back.p == p) idx = k == back.k + 1 ? 0 : 2;   // we are the region below / above it on the same branch
      else if (back.p > p) idx = 2;                     // it is one of our children: we are its "up"
      else idx = p == back.p + 1 ? 0 : 1;               // it is our parent: we are its children[1] / children[0]
      const int q = back.p;
      k = back.k;
      if (q != p) { load_node(q); if (size <= 1) size_c1 = 1; }
      next = idx + 1;
    }
  }
  if (overflow) { if (lane == 0) S.error = kSprErrFrontierCap; return; }
  __syncwarp();
  if (lane != 0) return;
  // ---- account_for_Xs_detachment (core/spr_study.cpp:130-209) + remove_regions_in_Xs_future (:211-224), in place -----------------------------
  const int root_id = f.node_id[root];
  const bool ccr = S.can_change_root != 0;
  int w = 0;
  if (posX < 0) {
    for (int i = 0; i < n_out; ++i) {
      RegionHead h = out[i];
      if (!ccr && h.branch == root_id) continue;
      if (h.t_min >= tX) continue;
      if (h.t_max > tX) h.t_max = tX;
      out[w++] = h;
    }
  } else {
    const int nP = S.nP, nS = S.nS;
    const int P_id = f.node_id[posP], S_id = f.node_id[posS];
    const bool P_is_root = S.P_is_root != 0;
    double tmin_P_last = 0.0;                            // region_t_min(P, nP): start of P's bottom region
    if (!P_is_root) tmin_P_last = nP == 0 ? f.t[f.parent_pos[posP]] : f.mut_t[f.mut_off[posP] + nP - 1];
    for (int i = 0; i < n_out; ++i) {
      RegionHead h = out[i];
      bool keep = true;
      if (!ccr && h.branch == root_id) keep = false;
      else if (h.branch == S_id || h.branch == P_id) {
        if (!P_is_root) {
          if (h.branch == S_id) { if (h.mut_idx == 0) h.t_min = tmin_P_last; h.mut_idx += nP; }
          else if (h.mut_idx == nP) keep = false;
          else h.branch = S_id;
        } else if (!ccr) {
          if (h.branch == P_id) keep = false;
        } else {
          if (h.branch == S_id && h.mut_idx == nS) { h.mut_idx += nP; h.t_min = -DBL_MAX; }
          else keep = false;
        }
      }
      if (!keep) continue;
      if (h.t_min >= tX) continue;
      if (h.t_max > tX) h.t_max = tX;
      out[w++] = h;
    }
  }
  S.total_regions = w;
}
