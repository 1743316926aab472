// kernels_spr_group2.cuh -- full SPR studies of ONE tree, 32 at a time, as a flat scan over mutation EVENTS and a flat emit over
// region TEMPLATES.  (included by kernels_spr.cu inside namespace dphy; replaces spr_gscan / spr_gemit of kernels_spr_group.cuh)
//
// What depends on the tree alone is tabulated once per forest (spr_tab_* kernels, cached in dphy_forest::d_spr_*):
//   * region templates: the regions (q, k), k = 0 .. np(q), of every node q in device (DFS) order -- N + M per tree; template index
//     of (q, k) = q + (mut_off[q] - mut_base) + k; tnode[] maps a template back to its node.
//   * events: walking the tree in DFS order, "enter" events (one per mutation of q, when q opens) and "exit" events (the same
//     mutations again when q's subtree closes) -- 2 M per tree.  The nodes closing right before position q are a contiguous slice of
//     the post-order list, so with PM = prefix of np over the post-order list the event index at which q opens is
//     eopen(q) = (mut_off[q] - mut_base) + PM[q - depth(q)], and the exits of a node with post-order index j, closing right before
//     position c, start at (mut_off[c] - mut_base) + PM[j].
// With d(m, s) the potential of mutation m for study s (kernels_spr.cu header) and S[e] = sum of +-d over the events before e, the
// Hamming potential at region (q, k) is simply S[eopen(q) + k]: the tree prefix sum with its closer correction becomes ONE plain
// prefix sum over events, the same for every node shape.
//
//   spr_g2_scan_kernel    lanes = studies.  A warp takes 128 consecutive events: event records loaded 32 at a time (coalesced) and
//                         broadcast, one 32-byte row of xT[site][32] gathered per event, chunk-local prefix stored as int8 rows
//                         S[e][32] (|prefix| <= 127 inside a chunk) + the chunk total.
//   spr_g2_emit_kernel<1> lanes = templates.  A warp takes 32 consecutive templates and loops over the 32 studies: keep flag of every
//                         (template, study) -> one ballot = the 32-bit keep mask of (chunk, study), stored with its popcount.
//   spr_g2_prefix_kernel  exclusive prefixes of the chunk totals (events) and of the kept counts (templates), per study.
//   (spr_segments_kernel lays out the DFS segments of every study from these and emits the special nodes: root, P, S, path nodes)
//   spr_g2_emit_kernel<0> the same loop again: rank inside the mask -> output index; the kept lanes of a warp write CONSECUTIVE
//                         32-byte heads of one study's array, so every store instruction covers whole lines and nothing is staged.
constexpr int kEvChunk = 128;      // events per warp of the scan (int8 chunk-local prefixes)
constexpr int kG2Warps = 4;

// ---- study-independent tables -----------------------------------------------------------------------------------------------------------
// PM[j] = number of mutations of the first j nodes of the tree's post-order list.  Two levels: every CTA scans one tile of 8,192
// entries (tile-local exclusive prefix + the tile total); the consumer adds the totals of the tiles before (a few dozen per tree).
constexpr int kPmTile = 1024 * 8;
__global__ void __launch_bounds__(1024) spr_tab_pm_kernel(ForestDev f, int32_t* __restrict__ PM, int32_t* __restrict__ tile_tot, int max_tiles) {
  __shared__ int s_ws[32];
  const TreeDev T = f.trees[blockIdx.y];
  const int nb = T.node_base, N = T.num_nodes;
  const int j0 = blockIdx.x * kPmTile;
  if (j0 >= N) return;
  int v[8], mine = 0;
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const int j = j0 + (int)threadIdx.x * 8 + u;
    v[u] = 0;
    if (j < N) { const int a = f.post_node[nb + j]; v[u] = f.mut_off[a + 1] - f.mut_off[a]; }
    mine += v[u];
  }
  int tot;
  const int incl = block_scan_incl<int, 1024>(mine, s_ws, &tot);
  int run = incl - mine;
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const int j = j0 + (int)threadIdx.x * 8 + u;
    if (j < N) PM[nb + j] = run;
    run += v[u];
  }
  if (threadIdx.x == 0) tile_tot[(size_t)blockIdx.y * max_tiles + blockIdx.x] = tot;
}

// eopen, tnode and the event list: one thread per node (grid.y = tree)
__global__ void __launch_bounds__(256) spr_tab_fill_kernel(ForestDev f, const int32_t* __restrict__ PM, const int32_t* __restrict__ tile_tot, int max_tiles,
                                                           int32_t* __restrict__ eopen, int32_t* __restrict__ tnode, int32_t* __restrict__ ev) {
  const TreeDev T = f.trees[blockIdx.y];
  const int nb = T.node_base, N = T.num_nodes;
  const int q = blockIdx.x * 256 + threadIdx.x;
  if (q >= N) return;
  const int p = nb + q;
  const int mb = f.mut_off[nb];
  const int moff = f.mut_off[p] - mb, np = f.mut_off[p + 1] - f.mut_off[p];
  const int dep = f.depth[p], size = f.subtree_size[p];
  const int32_t* tt = tile_tot + (size_t)blockIdx.y * max_tiles;
  auto pm_at = [&](int j) {                      // PM[j] = tile-local prefix + totals of the tiles before
    int s = PM[nb + j];
    for (int t = 0; t < j / kPmTile; ++t) s += __ldg(tt + t);
    return s;
  };
  const int eo = moff + pm_at(q - dep);
  eopen[p] = eo;
  int32_t* tn = tnode + (size_t)nb + mb + q + moff;          // global template base of the tree = nb + mb
  for (int k = 0; k <= np; ++k) tn[k] = p;
  if (np > 0) {
    int32_t* evt = ev + 2 * (size_t)mb;
    const int xo = (f.mut_off[p + size] - mb) + pm_at(q + size - 1 - dep);     // post-order index of q = q + size - 1 - depth
    for (int k = 0; k < np; ++k) { evt[eo + k] = moff + k; evt[xo + k] = (moff + k) | (int)0x80000000; }
  }
}

// ---- scan over events -------------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kG2Warps * 32) spr_g2_scan_kernel(ForestDev f, SprBatchDev B, const SprGroupDev* __restrict__ groups) {
  const unsigned full = 0xffffffffu;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const SprGroupDev& G = groups[blockIdx.y];
  const int chunk = blockIdx.x * kG2Warps + warp;
  if (chunk >= G.num_ev_chunks) return;
  const int nb = G.node_base, mb = G.mut_base, M2 = 2 * G.num_muts;
  const int np_root = f.mut_off[nb + 1] - f.mut_off[nb];       // the root's own list is never crossed: its events carry no potential
  const uint8_t* __restrict__ xT = (const uint8_t*)(B.slab + G.off_xT);
  int8_t* __restrict__ Srow = (int8_t*)(B.slab + G.off_S);
  const int32_t* __restrict__ ev = B.g2_ev + 2 * (size_t)mb;
  const int e0 = chunk * kEvChunk;
  int acc = 0;
#pragma unroll 1
  for (int b = 0; b < kEvChunk / 32; ++b) {
    // lane i holds event e0 + 32 b + i: (site, from|to, sign) -- pk bit 5 = carries a potential, bit 4 = exit
    const int e = e0 + b * 32 + lane;
    int site = 0, pk = 0;
    if (e < M2) {
      const int evv = __ldg(ev + e);
      const int mr = evv & 0x7fffffff;
      if (mr >= np_root) { site = __ldg(f.mut_site + mb + mr); pk = (__ldg(f.mut_code + mb + mr) & 15) | (evv < 0 ? 16 : 0) | 32; }
    }
#pragma unroll 8
    for (int i = 0; i < 32; ++i) {
      const int si = __shfl_sync(full, site, i), pi = __shfl_sync(full, pk, i);
      Srow[(size_t)(e0 + b * 32 + i) * kGroup + lane] = (int8_t)acc;        // one 32-byte sector per event
      if (pi & 32) {
        const int d = g_mut_dh(xT[(size_t)si * kGroup + lane], pi & 15);
        acc += (pi & 16) ? -d : d;
      }
    }
  }
  ((int32_t*)(B.slab + G.off_aggS))[(size_t)chunk * kGroup + lane] = acc;
}

// ---- exclusive prefixes over the chunk rows of a group: [rows][32] -> in place, totals in row [rows] ---------------------------------------
// A thread-block cluster of 8 CTAs per (group, table): CTA r owns a contiguous eighth of the rows (warp w a 32nd of that), sums it,
// publishes its column totals into the shared memory of every CTA of the cluster (distributed shared memory) and, after one cluster
// barrier, rewrites its rows as exclusive prefixes.  grid = (8, groups); one launch per table (the kept counts on the side stream).
constexpr int kPfxCtas = 8;
__global__ void __cluster_dims__(kPfxCtas, 1, 1) __launch_bounds__(1024) spr_g2_prefix_kernel(SprBatchDev B, const SprGroupDev* __restrict__ groups, int which) {
  __shared__ int s_w[32][33];                 // per-warp column sums of this CTA
  __shared__ int s_cta[kPfxCtas][32];         // column totals of every CTA of the cluster
  namespace cgx = cooperative_groups;
  cgx::cluster_group cluster = cgx::this_cluster();
  const int rank = (int)cluster.block_rank();
  const SprGroupDev& G = groups[blockIdx.y];
  const int rows = which == 0 ? G.num_ev_chunks : G.num_t_chunks + 1;      // which: 0 = event-chunk totals, 1 = kept counts
  int32_t* a = (int32_t*)(B.slab + (which == 0 ? G.off_aggS : G.off_aggK));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int per = (rows + kPfxCtas * 32 - 1) / (kPfxCtas * 32);
  const int r0 = min((rank * 32 + warp) * per, rows), r1 = min(r0 + per, rows);
  int sum = 0;
#pragma unroll 8
  for (int r = r0; r < r1; ++r) sum += a[(size_t)r * kGroup + lane];
  s_w[warp][lane] = sum;
  __syncthreads();
  if (warp < kPfxCtas) {
    // warp w of every CTA posts this CTA's column totals into CTA w
    int tot = 0;
#pragma unroll
    for (int w = 0; w < 32; ++w) tot += s_w[w][lane];
    *cluster.map_shared_rank(&s_cta[rank][lane], warp) = tot;
  }
  cluster.sync();
  int run = 0;
  for (int c = 0; c < rank; ++c) run += s_cta[c][lane];
  for (int w = 0; w < warp; ++w) run += s_w[w][lane];
#pragma unroll 4
  for (int r = r0; r < r1; ++r) {
    const int v = a[(size_t)r * kGroup + lane];
    a[(size_t)r * kGroup + lane] = run;
    run += v;
  }
  if (rank == kPfxCtas - 1 && warp == 31) a[(size_t)rows * kGroup + lane] = run;     // its (possibly empty) range ends at `rows`
}

// ---- keep masks (kCount) / emit over templates ---------------------------------------------------------------------------------------------
// What a template is, independent of the study: written once per batch and tree (spr_g2_templ_kernel), so that the two template
// kernels start from one 48-byte record per lane instead of a three-level chain of gathers through the node arrays.
struct alignas(16) G2Templ {
  double t_min, t_max;            // (t_min, t_max] of region (q, k) before any clipping; the root's t_min is unused
  int idn, k, q, qend;            // host node id, mutation index, tree-local position, end of the node's subtree
  int e, nonroot, moff, np;       // event-prefix row of the region; parent exists; the node's list (global offset, length)
};
// What the template loop needs of a study: constants of the batch (spr_g2_consts_kernel, after the X tables) ...
struct alignas(16) G2Const {
  double tX; int qX, xe;          // X's subtree = [qX, xe) in tree-local positions (empty when X is detached); tX = -DBL_MAX: dead lane
  int qS, qP, q0, cap;            // S, P, the start node; region capacity
};
// ... and what is known once the segments are laid out (spr_g2_bases_kernel)
struct alignas(16) G2Out {
  int mH, fused; unsigned long long out;     // init_min_muts - H0; weights computed by the emit; the study's head array
  double logfl, fa, lam, mu3;                // log(f lambda_X), f, lambda_X, mu / 3   (Spr_study::Spr_study, core/spr_study.cpp:239,313-318)
  long long lw_minus_out, pad;               // raw log-weight array relative to the head array, in bytes
};
struct alignas(16) G2Study { G2Const c; int base, mH; unsigned out_lo, out_hi; };
struct alignas(16) G2Weight { double logfl, fa, lam, mu3; long long lw_minus_out; int fused, pad; };
static_assert(sizeof(G2Templ) == 48 && sizeof(G2Const) == 32 && sizeof(G2Out) == 64 && sizeof(G2Study) == 48, "record sizes are part of the slab layout");

// Besides the records, per chunk of 32 templates (study-independent as well): the start times of its live templates SORTED
// (csort), the running OR of their lane bits in that order (cpm) and the chunk's first / last position (cq).  A region is kept iff it
// starts before t_X, so the keep mask of (chunk, study) is cpm[#{sorted starts < t_X} - 1]: the count kernel finds it with a
// five-step binary search per study, all 32 studies at once, instead of 32 x 32 comparisons.
__global__ void __launch_bounds__(256) spr_g2_templ_kernel(ForestDev f, SprBatchDev B, const SprGroupDev* __restrict__ groups) {
  const unsigned full = 0xffffffffu;
  const SprGroupDev& G = groups[blockIdx.y];
  if (!G.trec_owner) return;                       // one group per tree writes the records; the others share them
  const int r = blockIdx.x * 256 + threadIdx.x;
  const int tc = r >> 5, lane = threadIdx.x & 31;
  if (tc > G.num_t_chunks) return;                 // (whole warps)
  const int nb = G.node_base, mb = G.mut_base;
  const bool valid = r < G.num_templates;
  G2Templ T;
  T.t_min = DBL_MAX; T.t_max = DBL_MAX; T.idn = 0; T.k = 0; T.q = -3; T.qend = -3; T.e = 0; T.nonroot = 0; T.moff = 0; T.np = 0;
  if (valid) {
    const int p = __ldg(B.g2_tnode + (size_t)nb + mb + r);
    const int q = p - nb;
    const int moff = f.mut_off[p], np = f.mut_off[p + 1] - moff;
    const int k = r - (q + (moff - mb));
    const int par = f.parent_pos[p];
    T.nonroot = par >= 0;
    const double tn = f.t[p], tp = T.nonroot ? f.t[par] : 0.0;
    T.t_min = k == 0 ? tp : f.mut_t[moff + k - 1];
    T.t_max = k >= np ? tn : f.mut_t[moff + k];
    T.idn = f.node_id[p]; T.k = k; T.q = q; T.qend = q + f.subtree_size[p];
    T.e = B.g2_eopen[p] + k; T.moff = moff; T.np = np;
    ((G2Templ*)(B.slab + G.off_trec))[r] = T;
  }
  // bitonic sort of (start time, lane) over the warp; templates that can never be kept by the time rule (the root's, the padding of
  // the last chunk) sort last with the key DBL_MAX and contribute no bit
  double key = (valid && T.nonroot) ? T.t_min : DBL_MAX;
  int idx = lane;
#pragma unroll
  for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      const double ok = __shfl_xor_sync(full, key, j);
      const int oi = __shfl_xor_sync(full, idx, j);
      const bool keep_min = ((lane & j) == 0) == ((lane & k) == 0);
      const bool other_less = ok < key || (ok == key && oi < idx);
      if (keep_min == other_less) { key = ok; idx = oi; }
    }
  }
  unsigned pm = key != DBL_MAX ? (1u << idx) : 0u;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const unsigned u = __shfl_up_sync(full, pm, o); if (lane >= o) pm |= u; }
  ((double*)(B.slab + G.off_csort))[(size_t)tc * 32 + lane] = key;
  ((uint32_t*)(B.slab + G.off_cpm))[(size_t)tc * 32 + lane] = pm;
  const int nv = min(32, G.num_templates - tc * 32);
  const int qfirst = __shfl_sync(full, T.q, 0), qlast = __shfl_sync(full, T.q, max(nv - 1, 0));
  if (lane == 0) ((int2*)(B.slab + G.off_cq))[tc] = nv > 0 ? make_int2(qfirst, qlast) : make_int2(-3, -3);
}

__global__ void spr_g2_consts_kernel(ForestDev f, SprBatchDev B, const SprGroupDev* __restrict__ groups) {
  const SprGroupDev& G = groups[blockIdx.x];
  const int lane = threadIdx.x;
  const int nb = G.node_base;
  G2Const c;
  c.tX = -DBL_MAX; c.qX = -1; c.xe = -1; c.qS = -1; c.qP = -1; c.q0 = 0; c.cap = 0;
  if (lane < G.num) {
    const SprStudy& S = B.studies[G.study[lane]];
    if (!S.error) {
      c.tX = S.t_X;
      if (S.posX >= 0) { c.qX = S.posX - nb; c.xe = S.posX - nb + f.subtree_size[S.posX]; c.qS = S.posS - nb; c.qP = S.posP - nb; }
      c.q0 = S.pos0 - nb; c.cap = S.region_cap;
    }
  }
  ((G2Const*)(B.slab + G.off_consts))[lane] = c;
  // the root has ONE region, (root, np), kept iff the root may change and the root is not P (eval_region); it starts at -DBL_MAX
  int rk = 0;
  if (lane < G.num) { const SprStudy& S = B.studies[G.study[lane]]; rk = (!S.error && S.can_change_root && S.posP != S.root_pos) ? 1 : 0; }
  ((int32_t*)(B.slab + G.off_consts + 32 * kGroup))[lane] = rk;
}

// ---- per (chunk, study): where the chunk's kept regions go -------------------------------------------------------------------------------
// The regions of an off-path node go to  hang[j] + KB(node) + rank,  j = the deepest node of the study's start->root path that
// contains the node.  j is constant over long runs of positions, so it is found ONCE per (template chunk, study) here -- one thread
// each, the binary search over the study's nested path ranges running out of L1 (every thread of a CTA searches the same study) --
// instead of in the emit kernel's prologue, where ten dependent loads per warp were its critical path.  A chunk whose positions
// straddle a segment boundary of the study (at most two per path node) gets a row of per-template offsets instead, filled by the
// whole warp, one lane per template.
__device__ __forceinline__ int g2_classify(const int2* __restrict__ pae, int path_len, int p, int lo = 0, int hi = -1) {
  if (hi < 0) hi = path_len - 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const int2 ae = __ldg(pae + mid);
    if (p >= ae.x && p < ae.y) hi = mid; else lo = mid + 1;
  }
  return lo;
}

constexpr int kBasesPathSmem = 2048;      // path nodes whose ranges / offsets are staged in shared memory (deeper paths are read in place)
constexpr int kBasesThreads = 256, kBasesSlices = 16;
__global__ void __launch_bounds__(kBasesThreads) spr_g2_bases_kernel(SprBatchDev B, const SprGroupDev* __restrict__ groups) {
  __shared__ int2 s_pae[kBasesPathSmem];
  __shared__ int s_hang[kBasesPathSmem];
  const SprGroupDev& G = groups[blockIdx.y];
  const int s = blockIdx.x;
  if (s >= G.num) return;
  const int sidx = G.study[s];
  SprStudy& S = B.studies[sidx];
  if (S.error) return;
  const int nb = G.node_base, NT = G.num_templates;
  const G2Templ* __restrict__ trec = (const G2Templ*)(B.slab + G.off_trec);
  const int path_len = S.path_len;
  const int2* pae = (const int2*)(B.slab + S.off_pae);
  const int32_t* hang = (const int32_t*)(B.slab + S.off_hang);
  if (path_len <= kBasesPathSmem) {
    for (int i = threadIdx.x; i < path_len; i += kBasesThreads) { s_pae[i] = pae[i]; s_hang[i] = hang[i]; }
    pae = s_pae; hang = s_hang;
  }
  if (threadIdx.x == 0 && blockIdx.z == 0) {
    G2Out o; o.mH = S.init_min_muts - S.H0; o.fused = S.weights_fused; o.out = (unsigned long long)(B.slab + S.off_regions);
    o.logfl = log(S.f * S.lambda_X); o.fa = S.f; o.lam = S.lambda_X; o.mu3 = S.mu / 3;
    o.lw_minus_out = (long long)(S.off_lw - S.off_regions); o.pad = 0;
    ((G2Out*)(B.slab + G.off_outs))[s] = o;
  }
  __syncthreads();
  const uint32_t* __restrict__ maskcol = (const uint32_t*)(B.slab + G.off_mask) + s;
  const int32_t* __restrict__ aggKcol = (const int32_t*)(B.slab + G.off_aggK) + s;
  int2* cbase = (int2*)(B.slab + G.off_cbase) + s;
  int32_t* hmix = (int32_t*)(B.slab + S.off_hmix);
  const int pos0 = S.pos0;
  auto classify = [&](int p, int lo, int hi) {
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      const int2 ae = pae[mid];
      if (p >= ae.x && p < ae.y) hi = mid; else lo = mid + 1;
    }
    return lo;
  };
  // the study's chunks are split over gridDim.z CTAs; a warp takes 32 consecutive chunks per round
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int per = ((G.num_t_chunks + 1 + (int)gridDim.z - 1) / (int)gridDim.z + 31) & ~31;
  const int c0 = (int)blockIdx.z * per, c1 = min(c0 + per, G.num_t_chunks + 1);
  // (consecutive chunks go to different warps: straddling chunks cluster along the path, and each costs its warp a serial step)
  constexpr int kW = kBasesThreads / 32;
  const int wrp = threadIdx.x >> 5;
  for (int tb = c0; tb < c1; tb += kBasesThreads) {
    const int tc = tb + lane * kW + wrp;
    bool mixed = false;
    int jlo = 0, jhi = 0, kb = 0;
    if (tc < c1) {
      // (all four loads issued together: the chunk's first / last position come from the study-independent chunk records)
      const uint32_t mask = maskcol[(size_t)tc * kGroup];
      kb = aggKcol[(size_t)tc * kGroup];
      const int2 qfl = ((const int2*)(B.slab + G.off_cq))[tc];
      if (mask == 0u) cbase[(size_t)tc * kGroup] = make_int2(0, 0);
      else {
        const int pfirst = nb + qfl.x, plast = nb + qfl.y;
        const int j = classify(pfirst, 0, path_len - 1);
        const int2 cur = pae[j];
        const int dnx = j > 0 ? pae[j - 1].x : INT_MAX;
        mixed = (plast >= cur.y) || (dnx > pfirst && dnx <= plast);
        if (!mixed) cbase[(size_t)tc * kGroup] = make_int2(hang[j] + kb, 0);
        else {
          // the path index is monotone in the position on either side of the start node (and 0 inside its subtree): this brackets
          // the search of every template of the chunk
          const int jl = classify(plast, 0, path_len - 1);
          jlo = (pos0 >= pfirst && pos0 <= plast) ? 0 : min(j, jl);
          jhi = max(j, jl);
        }
      }
    }
    // chunks that straddle a segment boundary of the study: a row of 32 per-template offsets each, one lane per template; the
    // warp reserves its rows with one atomic
    unsigned todo = __ballot_sync(full, mixed);
    if (todo) {
      int row0 = 0;
      if (lane == 0) row0 = (int)atomicAdd(B.ticket + sidx * 4 + 3, (unsigned)__popc(todo));
      row0 = __shfl_sync(full, row0, 0);
      if (row0 + __popc(todo) > S.hmix_cap) { if (lane == 0) S.error = kSprErrHmixCap; todo = 0u; }
      for (int nrow = 0; todo; todo &= todo - 1, ++nrow) {
        const int src = __ffs(todo) - 1;
        const int tcs = tb + src * kW + wrp, lo_s = __shfl_sync(full, jlo, src), hi_s = __shfl_sync(full, jhi, src), kb_s = __shfl_sync(full, kb, src);
        const int row = row0 + nrow;
        const int r = tcs * 32 + lane;
        int h = 0;
        if (r < NT) h = hang[classify(nb + trec[r].q, lo_s, hi_s)];
        hmix[(size_t)row * 32 + lane] = h + kb_s;
        if (lane == src) cbase[(size_t)tcs * kGroup] = make_int2(row, 1);
      }
    }
  }
}

__device__ __noinline__ bool g2_special_keep(const ForestDev& f, const SprBatchDev& B, int sidx, int p, int k, int np, int moff) {
  const int par = f.parent_pos[p];
  return eval_region(f, B.studies[sidx], p, k, np, moff, par >= 0 ? f.t[par] : 0.0, f.t[p]).keep;
}

// ---- keep masks + kept counts of every (template chunk, study): lanes = studies -----------------------------------------------------------
constexpr int kCountWarps = 8, kCountPerWarp = 8;     // chunks per CTA = 64: the per-chunk work is ~100 instructions, CTA launch would dominate
__global__ void __launch_bounds__(kCountWarps * 32) spr_g2_count_kernel(ForestDev f, SprBatchDev B, const SprGroupDev* __restrict__ groups) {
  const unsigned full = 0xffffffffu;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const SprGroupDev& G = groups[blockIdx.y];
  const int nb = G.node_base, NT = G.num_templates;
  const G2Const c = ((const G2Const*)(B.slab + G.off_consts))[lane];
  const int r_root = f.mut_off[nb + 1] - f.mut_off[nb];          // template index of the root's one region, (root, np)
#pragma unroll 2
  for (int it = 0; it < kCountPerWarp; ++it) {
  const int tc = (blockIdx.x * kCountWarps + warp) * kCountPerWarp + it;
  if (tc > G.num_t_chunks) return;                    // chunk num_t_chunks exists (empty): KB(N) reads its row
  const double sorted = ((const double*)(B.slab + G.off_csort))[(size_t)tc * 32 + lane];
  const unsigned pm = ((const uint32_t*)(B.slab + G.off_cpm))[(size_t)tc * 32 + lane];
  const int2 qfl = ((const int2*)(B.slab + G.off_cq))[tc];
  // number of the chunk's sorted start times before this lane's t_X (binary lifting over the warp's registers)
  int n = 0;
#pragma unroll
  for (int step = 16; step >= 1; step >>= 1) { const double v = __shfl_sync(full, sorted, n + step - 1); if (v < c.tX) n += step; }
  { const double v = __shfl_sync(full, sorted, 31); if (n == 31 && v < c.tX) n = 32; }
  const unsigned pmn = __shfl_sync(full, pm, max(n - 1, 0));
  uint32_t mymask = n > 0 ? pmn : 0u;
  const int qfirst = qfl.x, qlast = qfl.y;
  if (qfirst >= c.qX && qlast < c.xe) mymask = 0u;          // the whole chunk lies inside X's subtree
  if (tc == (r_root >> 5)) mymask |= (uint32_t)((const int32_t*)(B.slab + G.off_consts + 32 * kGroup))[lane] << (r_root & 31);
  // S and P (relabelled by account_for_Xs_detachment) follow the general rules, as in node_kept_count; a chunk that holds one of
  // them for some study, or an end of that study's X subtree, is redone for that study template by template
  const bool has_special = c.tX != -DBL_MAX && qfirst >= 0 &&
                           ((c.qS >= qfirst && c.qS <= qlast) || (c.qP >= qfirst && c.qP <= qlast) ||
                            (c.qX > qfirst && c.qX <= qlast) || (c.xe > qfirst && c.xe <= qlast));
  unsigned specmask = __ballot_sync(full, has_special);
  if (specmask) {
    const int r = tc * 32 + lane;
    const bool valid = r < NT;
    G2Templ T;
    T.t_min = DBL_MAX; T.k = 0; T.q = -3; T.nonroot = 0; T.moff = 0; T.np = 0;
    if (valid) {
      const uint4* tp = reinterpret_cast<const uint4*>((const G2Templ*)(B.slab + G.off_trec) + r);
      const uint4 a = __ldg(tp), b = __ldg(tp + 1), cc = __ldg(tp + 2);
      T.t_min = __hiloint2double(a.y, a.x); T.k = b.y; T.q = b.z; T.nonroot = cc.y; T.moff = cc.z; T.np = cc.w;
    }
    const bool nonroot = T.nonroot != 0;
    const int q = T.q;
    for (; specmask; specmask &= specmask - 1u) {
      const int s = __ffs(specmask) - 1;
      const double tX = __shfl_sync(full, c.tX, s);
      const int qX = __shfl_sync(full, c.qX, s), xe = __shfl_sync(full, c.xe, s), qS = __shfl_sync(full, c.qS, s), qP = __shfl_sync(full, c.qP, s);
      bool keep = valid && nonroot && T.t_min < tX && !(q >= qX && q < xe);
      if (valid && (q == qS || q == qP || !nonroot)) {
        keep = false;
        if (nonroot || T.k == T.np) keep = g2_special_keep(f, B, G.study[s], nb + q, T.k, T.np, T.moff);
      }
      const unsigned bal = __ballot_sync(full, keep);
      if (lane == s) mymask = bal;
    }
  }
  ((uint32_t*)(B.slab + G.off_mask))[(size_t)tc * kGroup + lane] = mymask;
  ((int32_t*)(B.slab + G.off_aggK))[(size_t)tc * kGroup + lane] = __popc(mymask);
  }
}

// ---- emit: lanes = templates, loop over the studies ------------------------------------------------------------------------------------------
// the 32-byte heads, and the raw log-weights (and their per-study maximum) of the studies with weights_fused
__global__ void __launch_bounds__(kG2Warps * 32) spr_g2_emit_kernel(ForestDev f, SprBatchDev B, const SprGroupDev* __restrict__ groups) {
  __shared__ G2Study s_st[kG2Warps][kGroup];
  __shared__ G2Weight s_wt[kG2Warps][kGroup];
  __shared__ double2 s_log[1 << kLogTabBits];
  // chunk-local potentials of the lane's template for the 32 studies: one 32-byte row, kept in shared memory (36-byte pitch) because
  // the study loop is not fully unrolled -- 32 copies of its body, two logarithms each, do not fit the instruction cache: ncu showed
  // "no instruction" as the top stall -- so the byte of study s is a dynamic index
  __shared__ uint32_t s_row[kG2Warps][32][9];
  fill_log_table(s_log);
  __syncthreads();
  const unsigned full = 0xffffffffu;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const SprGroupDev& G = groups[blockIdx.y];
  const int tc = blockIdx.x * kG2Warps + warp;
  if (tc >= G.num_t_chunks) return;
  const int NT = G.num_templates;

  // ---- the lane's study (everything one level deep) -----------------------------------------------------------------------------------
  G2Study st;
  st.c = ((const G2Const*)(B.slab + G.off_consts))[lane];
  uint32_t mymask = ((const uint32_t*)(B.slab + G.off_mask))[(size_t)tc * kGroup + lane];
  const int2 cb = ((const int2*)(B.slab + G.off_cbase))[(size_t)tc * kGroup + lane];
  const G2Out* op = (const G2Out*)(B.slab + G.off_outs) + lane;
  const int4 o0 = *reinterpret_cast<const int4*>(op);
  st.base = cb.x; st.mH = o0.x; st.out_lo = (unsigned)o0.z; st.out_hi = (unsigned)o0.w;
  unsigned long long mykey = 0ULL;                        // running maximum of the lane's study, as an ordered key
  {
    G2Weight w; w.logfl = op->logfl; w.fa = op->fa; w.lam = op->lam; w.mu3 = op->mu3; w.lw_minus_out = op->lw_minus_out; w.fused = o0.y; w.pad = 0;
    s_wt[warp][lane] = w;
  }
  const bool fused_lane = o0.y != 0;                      // the lane's study gets its weights here
  // (the constants were written on the side stream, before the X-table kernel could flag its study: look at the study itself)
  if (st.c.tX == -DBL_MAX || (lane < G.num && B.studies[G.study[lane]].error)) mymask = 0u;
  // ---- the lane's template ---------------------------------------------------------------------------------------------------------------
  const int r = tc * 32 + lane;
  const bool valid = r < NT;
  G2Templ T;
  T.t_min = DBL_MAX; T.t_max = DBL_MAX; T.idn = 0; T.k = 0; T.q = -2; T.qend = -2; T.e = 0; T.nonroot = 0; T.moff = 0; T.np = 0;
  if (valid) {
    const uint4* tp = reinterpret_cast<const uint4*>((const G2Templ*)(B.slab + G.off_trec) + r);
    const uint4 a = __ldg(tp), b = __ldg(tp + 1), c = __ldg(tp + 2);
    T.t_min = __hiloint2double(a.y, a.x); T.t_max = __hiloint2double(a.w, a.z);
    T.idn = b.x; T.k = b.y; T.q = b.z; T.qend = b.w; T.e = c.x; T.nonroot = c.y; T.moff = c.z; T.np = c.w;
  }
  if (!__any_sync(full, mymask != 0u)) return;
  const bool nonroot = T.nonroot != 0;
  const int q = T.q;
  // the chunk prefixes of the event chunk of the warp's first template are folded into the study constants, the (few) lanes in a
  // later event chunk add the difference
  const uint4* rp = reinterpret_cast<const uint4*>(B.slab + G.off_S + (size_t)T.e * kGroup);
  {
    const uint4 row0 = __ldg(rp), row1 = __ldg(rp + 1);
    uint32_t* rw = s_row[warp][lane];
    rw[0] = row0.x; rw[1] = row0.y; rw[2] = row0.z; rw[3] = row0.w; rw[4] = row1.x; rw[5] = row1.y; rw[6] = row1.z; rw[7] = row1.w;
  }
  const int ec = T.e >> 7, ec0 = __shfl_sync(full, ec, 0);
  const int32_t* aggrow = (const int32_t*)(B.slab + G.off_aggS) + (size_t)ec * kGroup;
  const int32_t* aggrow0 = (const int32_t*)(B.slab + G.off_aggS) + (size_t)ec0 * kGroup;
  const bool uniform = __all_sync(full, !valid || ec == ec0);
  st.mH += aggrow0[lane];
  s_st[warp][lane] = st;
  __syncwarp();
  const unsigned lt = (1u << lane) - 1u;
  // log(t_max - t_min) of the unclipped region: shared by every study that does not clip it
  const double logdt = fast_log(T.t_max - T.t_min, s_log);
  const int8_t* myrow = reinterpret_cast<const int8_t*>(s_row[warp][lane]);

#pragma unroll 4
  for (int s = 0; s < kGroup; ++s) {
    const unsigned bal = __shfl_sync(full, mymask, s);
    if (bal == 0u) continue;
    const G2Study& ss = s_st[warp][s];
    const bool special = q == ss.c.qS || q == ss.c.qP || !nonroot || (q <= ss.c.q0 && ss.c.q0 < T.qend);
    const bool emit = ((bal >> lane) & 1u) && !special;
    int base = ss.base;
    if (__shfl_sync(full, cb.y, s)) {
      // a chunk that straddles a segment boundary of this study: per-template offsets (spr_g2_bases_kernel); base is the row
      const SprStudy& S = B.studies[G.study[s]];
      base = ((const int32_t*)(B.slab + S.off_hmix))[(size_t)base * 32 + lane];
    }
    const int idx = base + __popc(bal & lt);
    unsigned long long key = 0ULL;
    if (emit && idx >= 0 && idx < ss.c.cap) {
      int m = ss.mH + myrow[s];                             // chunk-local prefix of study s + everything folded into mH
      if (!uniform) m += __ldg(aggrow + s) - __ldg(aggrow0 + s);
      const double tmx = T.t_max > ss.c.tX ? ss.c.tX : T.t_max;
      char* o = (char*)(((unsigned long long)ss.out_hi << 32) | ss.out_lo) + (size_t)idx * sizeof(RegionHead);
      const unsigned long long w0 = (unsigned long long)(unsigned)T.idn | ((unsigned long long)(unsigned)T.k << 32);
      asm volatile("st.global.v4.b64 [%0], {%1, %2, %3, %4};" ::"l"(o), "l"(w0), "l"(__double_as_longlong(T.t_min)),
                   "l"(__double_as_longlong(tmx)), "l"((unsigned long long)(unsigned)m) : "memory");
      if (s_wt[warp][s].fused) {
        // raw log-weight (core/spr_study.cpp:313-318): log(f lam dt) + f (-lam (t_X - t') + m log(mu (t_X - t') / 3)), t' = mid-point
        const G2Weight& w8 = s_wt[warp][s];
        const double x = ss.c.tX - 0.5 * (T.t_min + tmx);
        const double ldt = T.t_max > ss.c.tX ? fast_log(ss.c.tX - T.t_min, s_log) : logdt;
        const double lw = (w8.logfl + ldt) + w8.fa * (-(w8.lam * x) + m * fast_log(w8.mu3 * x, s_log));
        *reinterpret_cast<double*>(o - (size_t)idx * sizeof(RegionHead) + w8.lw_minus_out + (size_t)idx * sizeof(double)) = lw;
        key = f64_order_key(lw);
      }
    }
    // warp maximum of the ordered keys (two 32-bit REDUX steps), kept by the lane that owns study s
    const unsigned hi = (unsigned)(key >> 32), mh = __reduce_max_sync(full, hi);
    const unsigned ml = __reduce_max_sync(full, hi == mh ? (unsigned)key : 0u);
    if (lane == s) { const unsigned long long k2 = ((unsigned long long)mh << 32) | ml; if (k2 > mykey) mykey = k2; }
  }
  if (fused_lane && mykey != 0ULL) atomicMax(&B.studies[G.study[lane]].max_key, mykey);
}
