// kernels_logg.cu -- EMAT log-G evaluation for a whole forest (sm_100a).
//
// Replaces, for every tree of the forest in ONE evaluation:
//   calc_lambda_i                          core/phylo_tree_calc.cpp:420-436  (+ phylo_tree_calc.h:121-155)
//   calc_num_sites_missing_at_every_node   core/phylo_tree_calc.cpp:67-76
//   calc_log_root_prior                    core/phylo_tree_calc.cpp:467-504
//   calc_log_G_below_root                  core/phylo_tree_calc.cpp:515-543  (+ phylo_tree_calc.h:185-206)
//   calc_num_muts / calc_num_muts_ab / calc_T   core/phylo_tree_calc.cpp:577-597, :120-128
//
// Formulation.  The reference computes lambda_i with a pre-order walk (lambda_child = lambda_parent + delta of the
// branch) and then sums branch terms in node-index order.  Here nodes are stored in DFS pre-order and the per-branch
// lists in CSR in that same order, so
//   * the events of consecutive nodes are consecutive in memory: every thread walks the short lists of its own two
//     nodes with batched, predicated loads and the warp as a whole still streams whole cache lines;
//   * D[q], the pre-order inclusive prefix of the branch deltas, is one block scan;
//   * the nodes whose subtree closes right before position q are the contiguous slice post_node[c(q-1) .. c(q)),
//     c(q) = q - depth[q], of the tree's post-order list, so the sum of the deltas of everything already closed is a
//     prefix over that list evaluated at c(q);
//   * lambda[q] = lambda_ref + D[q] - CL[c(q)]: two scans and two gathers.
// Each CTA owns a tile of kLgTile consecutive positions of one tree and works on tile-local prefixes (magnitudes stay
// O(tile), so differences of prefixes lose nothing that matters at the 1e-9 tolerance).  Closers that opened in an
// earlier tile ("straddlers": subtree closes in a later tile than it opens; listed once at upload) get their delta from a tiny
// pre-kernel, so no CTA ever waits for another one.  A one-CTA-per-tree kernel then scans the tile aggregates and
// folds log G = sum_tiles (A1 - prefix * A2).  lambda_i / nsmn stay on the device as (tile-local value, tile prefix): each
// is written exactly once per evaluation, and the getters add the two when the host asks for them.
// Fixed reduction shapes everywhere => bit-reproducible results.
#include "dphy_internal.h"
#include "device_utils.cuh"

#include <math_constants.h>
#include <algorithm>
#include <cstdlib>

namespace dphy {

struct LogGParams {
  ForestDev f;
  double* lambda_out;    // [num_nodes] device order
  int32_t* nsmn_out;     // [num_nodes] device order
  double* tile_agg;      // [num_ctiles] sum of diff over the tile; overwritten by the tile's exclusive prefix in pass 2
  int32_t* tile_iagg;
  double* tile_part;     // [num_ctiles * 2]  (A1 = sum[-(lambda_ref+incl) len + g], A2 = sum len)
  int32_t* tile_ipart;   // [num_ctiles * 17] (num_muts, num_muts_ab[16])
  double* tree_out;      // [num_trees * 4]: log_root_prior, log_G_below_root, T, lambda_root
  int32_t* tree_iout;    // [num_trees * 20]: num_muts, 0, num_muts_ab[16], 0, 0
  double* sd_delta;      // [num_nodes] delta-lambda of the straddlers (sparse)
  int32_t* sd_n;         // [num_nodes] missing-site count of the straddlers (sparse)
  const int32_t* strad_list;   // device positions of the straddlers
  int32_t num_strad;
};

constexpr int kNW = kLgThreads / 32;

// conflict-free smem slot of event s (each thread owns a run of consecutive events)
__device__ __forceinline__ int pad_idx(int s) { return s + (s >> 3); }

struct LogGSmem {
  double dl[kLgTile];          // delta-lambda of every node of the tile
  int dn[kLgTile];             // sites going missing on every branch of the tile
  double clx[kLgTile + 2];     // exclusive prefix over the current chunk of the tile's closer list
  int cln[kLgTile + 2];
  double wsd[kNW * 3];
  int wsi[kNW];
  int ab[4 * 16];
};

// Exclusive block scan of up to (double, double, int) with ONE barrier pair; totals returned to every thread.
template <bool kB, bool kC>
__device__ __forceinline__ void block_scan_excl3(double& a, double& b, int& c, double& ta, double& tb, int& tc, LogGSmem& sm) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double ia = a, ib = b; int ic = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double ua = __shfl_up_sync(0xffffffffu, ia, o);
    double ub = 0.0; int uc = 0;
    if (kB) ub = __shfl_up_sync(0xffffffffu, ib, o);
    if (kC) uc = __shfl_up_sync(0xffffffffu, ic, o);
    if (lane >= o) { ia += ua; if (kB) ib += ub; if (kC) ic += uc; }
  }
  if (lane == 31) { sm.wsd[warp * 3] = ia; if (kB) sm.wsd[warp * 3 + 1] = ib; if (kC) sm.wsi[warp] = ic; }
  __syncthreads();
  double pa = 0.0, pb = 0.0; int pc = 0;
  ta = 0.0; tb = 0.0; tc = 0;
#pragma unroll
  for (int w = 0; w < kNW; ++w) {          // fixed order: deterministic
    const double wa = sm.wsd[w * 3];
    if (w < warp) pa += wa;
    ta += wa;
    if (kB) { const double wb = sm.wsd[w * 3 + 1]; if (w < warp) pb += wb; tb += wb; }
    if (kC) { const int wc = sm.wsi[w]; if (w < warp) pc += wc; tc += wc; }
  }
  a = pa + ia - a; if (kB) b = pb + ib - b; if (kC) c = pc + ic - c;
  __syncthreads();                         // wsd / wsi may be rewritten by the next scan
}

// Sequential delta-lambda / missing-site count of ONE branch (phylo_tree_calc.h:121-155); used for the straddlers.
__device__ void branch_delta_seq(const ForestDev& f, const SitesDev& S, int p, double& delta, int& nmiss) {
  const bool uni = S.nu_uniform != 0;
  double dm = 0.0;
  for (int i = f.mut_off[p]; i < f.mut_off[p + 1]; ++i) {
    const int code = __ldg(f.mut_code + i), pt = code >> 4, x = (code >> 2) & 3, y = code & 3;
    const double mn = uni ? S.mu[pt] * S.nu_const : __ldg(S.munu + __ldg(f.mut_site + i));
    dm += mn * ((-S.q[pt * 16 + y * 5]) - (-S.q[pt * 16 + x * 5]));
  }
  double dmi = 0.0;
  int nm = 0;
  for (int i = f.miss_off[p]; i < f.miss_off[p + 1]; ++i) {
    const int2 se = __ldg(f.miss_se + i);
    dmi -= __ldg(S.cumQ + se.y) - __ldg(S.cumQ + se.x);
    nm += se.y - se.x;
  }
  for (int i = f.fs_off[p]; i < f.fs_off[p + 1]; ++i) {
    const int code = __ldg(f.fs_code + i), pt = code >> 4, x = (code >> 2) & 3, y = code & 3;
    const double mn = uni ? S.mu[pt] * S.nu_const : __ldg(S.munu + __ldg(f.fs_site + i));
    dmi -= mn * ((-S.q[pt * 16 + y * 5]) - (-S.q[pt * 16 + x * 5]));
  }
  delta = dm + dmi;
  nmiss = nm;
}

// ---- pass 0: deltas of the straddlers (nodes whose subtree closes in a later log-G tile than it opens) ------------------------
__global__ void __launch_bounds__(128) emat_log_G_straddler_kernel(const LogGParams P) {
  const int i = blockIdx.x * 128 + threadIdx.x;
  if (i >= P.num_strad) return;
  const int2 ent = __ldg(reinterpret_cast<const int2*>(P.strad_list) + i);     // (device position, sites table)
  double d; int n;
  branch_delta_seq(P.f, P.f.sites[ent.y], ent.x, d, n);
  P.sd_delta[ent.x] = d;
  P.sd_n[ent.x] = n;
}

// ---- pass 1 --------------------------------------------------------------------------------------------------------------------
// kLgTile consecutive device positions of one tree per tile; thread tid owns the two consecutive positions 2 tid and
// 2 tid + 1.  emat_log_G_tile_kernel: one CTA per tile straight from global memory, thread-per-node list walks with batched,
// predicated loads; any site-rate model.
constexpr int kIvlBatch = 4;   // missation intervals in flight per node per round
constexpr int kMutBatch = 2;   // mutations in flight per node per round

// 4 resident CTAs per SM: 64 registers, no spills (5 or 6 CTAs: 48 / 40 registers, 80 / 160 bytes of spill stores)
__global__ void __launch_bounds__(kLgThreads, 4) emat_log_G_tile_kernel(const LogGParams P, const int32_t* __restrict__ tile_list) {
  __shared__ LogGSmem sm;
  const ForestDev& f = P.f;
  const int tid = threadIdx.x;
  const int tile = tile_list[blockIdx.x];
  const int4 ct = __ldg(reinterpret_cast<const int4*>(f.ctiles + tile));
  const int4 cl = __ldg(reinterpret_cast<const int4*>(f.ctiles + tile) + 1);
  const int tile_start = ct.x, n_act = ct.y, node_base = ct.z, cl0 = cl.x, cl1 = cl.y;
  const SitesDev& S = f.sites[ct.w];
  const bool uni = S.nu_uniform != 0;
  const double* __restrict__ cumQ = S.cumQ;
  if (tid < 64) sm.ab[tid] = 0;

  // ---- node records ----------------------------------------------------------------------------------------------------------------
  const int q0 = 2 * tid, p0 = tile_start + q0;
  const bool act0 = q0 < n_act, act1 = q0 + 1 < n_act;
  int par[2], dep[2], nmiss[2], om[3] = {0, 0, 0}, oi[3] = {0, 0, 0}, of[3] = {0, 0, 0};
  double tN[2], tP[2], dm[2], es[2], dmi[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) { par[k] = -1; dep[k] = 0; tN[k] = 0.0; tP[k] = 0.0; dm[k] = 0.0; es[k] = 0.0; dmi[k] = 0.0; nmiss[k] = 0; }
  if (act0) {
    par[0] = f.parent_pos[p0]; dep[0] = f.depth[p0]; tN[0] = f.t[p0];
    om[0] = f.mut_off[p0]; oi[0] = f.miss_off[p0]; of[0] = f.fs_off[p0];
    om[1] = f.mut_off[p0 + 1]; oi[1] = f.miss_off[p0 + 1]; of[1] = f.fs_off[p0 + 1];
    om[2] = om[1]; oi[2] = oi[1]; of[2] = of[1];
  }
  if (act1) {
    par[1] = f.parent_pos[p0 + 1]; dep[1] = f.depth[p0 + 1]; tN[1] = f.t[p0 + 1];
    om[2] = f.mut_off[p0 + 2]; oi[2] = f.miss_off[p0 + 2]; of[2] = f.fs_off[p0 + 2];
  }
#pragma unroll
  for (int k = 0; k < 2; ++k) if (par[k] >= 0) tP[k] = f.t[par[k]];

  // ---- per-node sums over the branch lists (list order => deterministic) -----------------------------------------------------------
  // missation intervals: -(cumQ[end] - cumQ[start]); count of sites going missing
  {
    const int c0 = oi[1] - oi[0], c1 = oi[2] - oi[1];
    const int cmax = max(c0, c1);
    for (int j = 0; j < cmax; j += kIvlBatch) {
      int2 se[2][kIvlBatch];
#pragma unroll
      for (int u = 0; u < kIvlBatch; ++u) {
        se[0][u] = j + u < c0 ? __ldg(f.miss_se + oi[0] + j + u) : make_int2(0, 0);
        se[1][u] = j + u < c1 ? __ldg(f.miss_se + oi[1] + j + u) : make_int2(0, 0);
      }
#pragma unroll
      for (int u = 0; u < kIvlBatch; ++u) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          // (0,0) for an absent interval: cumQ[0] - cumQ[0] == 0 exactly, so the arithmetic stays branch-free
          dmi[k] -= __ldg(cumQ + se[k][u].y) - __ldg(cumQ + se[k][u].x);
          nmiss[k] += se[k][u].y - se[k][u].x;
        }
      }
    }
  }
  // mutations: d_i = mu nu (q_to - q_from);  e_i = d_i * t_i + log(mu nu q_from,to)   [g_node = sum e_i - t_P * sum d_i]
  {
    const int c0 = om[1] - om[0], c1 = om[2] - om[1];
    const int cmax = max(c0, c1);
    for (int j = 0; j < cmax; j += kMutBatch) {
#pragma unroll
      for (int u = 0; u < kMutBatch; ++u) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          if (j + u < (k == 0 ? c0 : c1)) {
            const int i = om[k] + j + u;
            const int code = __ldg(f.mut_code + i) & 63;
            const double tm = __ldg(f.mut_t + i);
            double dd, lg;
            if (uni) { dd = __ldg(S.tab_md + code); lg = __ldg(S.tab_lq + code); }
            else {
              // log(mu nu_l q_xy) = log(mu nu_l) [per site, tabulated with mu nu_l] + log(q_xy) [64-entry table]: one 16-byte gather
              // instead of an fp64 log per mutation (a third of this kernel's instructions with site-rate heterogeneity on)
              const double2 mn = __ldg(S.munu2 + __ldg(f.mut_site + i));
              dd = mn.x * __ldg(S.tab_dq + code);
              lg = ((code >> 2) & 3) != (code & 3) ? mn.y + __ldg(S.tab_logq + code) : 0.0;
            }
            dm[k] += dd;
            if (par[k] >= 0) {     // the root's list ("mutations" above the root) is not part of log G nor of the counts
              es[k] += dd * tm + lg;
              atomicAdd(&sm.ab[(tid & 3) * 16 + (code & 15)], 1);
            }
          }
        }
      }
    }
  }
  // from-state overrides of missing sites: folded per-branch state counts when the site rates are uniform, lists otherwise
  if (uni) {
    for (int k2 = 0; k2 < f.fsw_stride; ++k2) {
      const double mq = __ldg(S.tab_muq + k2);
      if (act0) dmi[0] += mq * (double)__ldg(f.fsw + (size_t)p0 * f.fsw_stride + k2);
      if (act1) dmi[1] += mq * (double)__ldg(f.fsw + (size_t)(p0 + 1) * f.fsw_stride + k2);
    }
  } else {
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      for (int i = of[k]; i < of[k + 1]; ++i) {
        const int code = __ldg(f.fs_code + i) & 63;
        dmi[k] -= __ldg(S.munu + __ldg(f.fs_site + i)) * __ldg(S.tab_dq + code);
      }
    }
  }

  const double lambda_ref = __ldg(cumQ + S.L);
  const int32_t* post = f.post_node + node_base;   // post[j], j in [cl0, cl1)
  const int q_first = tile_start - node_base;
  const double d0 = act0 ? dm[0] + dmi[0] : 0.0, d1 = act1 ? dm[1] + dmi[1] : 0.0;
  const int n0 = act0 ? nmiss[0] : 0, n1 = act1 ? nmiss[1] : 0;
  sm.dl[q0] = d0; sm.dl[q0 + 1] = d1;
  sm.dn[q0] = n0; sm.dn[q0 + 1] = n1;

  // ---- D = inclusive prefix of the deltas over the tile's positions ------------------------------------------------------------
  double D[2]; int Dn[2];
  {
    double a = d0 + d1, b = 0.0, ta, tb; int c = n0 + n1, tc2;
    block_scan_excl3<false, true>(a, b, c, ta, tb, tc2, sm);       // also publishes dl / dn to the whole CTA
    D[0] = a + d0; D[1] = D[0] + d1;
    Dn[0] = c + n0; Dn[1] = Dn[0] + n1;
  }

  // ---- closers: prefix over the tile's slice of the post-order list, gathered at c(q) = q - depth[q] --------------------------
  double CL[2] = {0.0, 0.0};
  int CLn[2] = {0, 0};
  {
    const int myc0 = act0 ? (q_first + q0) - dep[0] : cl0, myc1 = act1 ? (q_first + q0 + 1) - dep[1] : cl0;
    double carry = 0.0; int icarry = 0;
    for (int c0 = cl0; c0 < cl1; c0 += kLgTile) {
      double a[2] = {0.0, 0.0}; int n[2] = {0, 0};
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int j = c0 + 2 * tid + u;
        if (j < cl1) {
          const int p = __ldg(post + j);
          const int qa = p - tile_start;
          if (qa >= 0) { a[u] = sm.dl[qa]; n[u] = sm.dn[qa]; }
          else { a[u] = __ldg(P.sd_delta + p); n[u] = __ldg(P.sd_n + p); }     // straddler: opened in an earlier tile
        }
      }
      double sa = a[0] + a[1], sb = 0.0, ta, tb; int sc = n[0] + n[1], tc2;
      block_scan_excl3<false, true>(sa, sb, sc, ta, tb, tc2, sm);
      sm.clx[2 * tid] = carry + sa; sm.clx[2 * tid + 1] = carry + sa + a[0];
      sm.cln[2 * tid] = icarry + sc; sm.cln[2 * tid + 1] = icarry + sc + n[0];
      carry += ta; icarry += tc2;
      if (tid == 0) { sm.clx[kLgTile] = carry; sm.cln[kLgTile] = icarry; }
      __syncthreads();
      if (myc0 > c0 && myc0 <= c0 + kLgTile) { CL[0] = sm.clx[myc0 - c0]; CLn[0] = sm.cln[myc0 - c0]; }
      if (myc1 > c0 && myc1 <= c0 + kLgTile) { CL[1] = sm.clx[myc1 - c0]; CLn[1] = sm.cln[myc1 - c0]; }
      __syncthreads();
    }
  }

  // ---- tile-local lambda_i / nsmn (device order); per-tile partial sums ----------------------------------------------------------
  double contrib = 0.0, tcontrib = 0.0;
  int nmut = 0;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int q = q0 + k, p = tile_start + q;
    if (q < n_act) {
      const double loc = D[k] - CL[k];
      const int iloc = Dn[k] - CLn[k];
      const double lam_local = lambda_ref + loc;     // + the tile's prefix (tile_agg after pass 2)
      P.lambda_out[p] = lam_local;
      P.nsmn_out[p] = iloc;
      if (q == n_act - 1) { P.tile_agg[tile] = loc; P.tile_iagg[tile] = iloc; }
      if (par[k] >= 0) {
        const double len = tN[k] - tP[k];
        contrib += -lam_local * len + (es[k] - tP[k] * dm[k]);
        tcontrib += len;
        nmut += om[k + 1] - om[k];
      }
    }
  }
  // three sums with one barrier
  {
    const int lane = tid & 31, warp = tid >> 5;
    contrib = warp_sum(contrib); tcontrib = warp_sum(tcontrib); nmut = warp_sum(nmut);
    if (lane == 0) { sm.wsd[warp * 3 + 0] = contrib; sm.wsd[warp * 3 + 1] = tcontrib; sm.wsd[warp * 3 + 2] = (double)nmut; }
    __syncthreads();
    if (warp == 0) {
      double a = lane < kNW ? sm.wsd[lane * 3 + 0] : 0.0;
      double b = lane < kNW ? sm.wsd[lane * 3 + 1] : 0.0;
      double c = lane < kNW ? sm.wsd[lane * 3 + 2] : 0.0;
      a = warp_sum(a); b = warp_sum(b); c = warp_sum(c);
      if (lane == 0) {
        P.tile_part[tile * 2 + 0] = a;
        P.tile_part[tile * 2 + 1] = b;
        P.tile_ipart[tile * 17 + 0] = (int)c;
      }
    }
  }
  if (tid < 16) P.tile_ipart[tile * 17 + 1 + tid] = sm.ab[tid] + sm.ab[16 + tid] + sm.ab[32 + tid] + sm.ab[48 + tid];
}

// ---- pass 2: one CTA per tree -- exclusive scan of the tile aggregates (tile order), log G fold, tallies, root prior -----
constexpr int kTreeThreads = 1024;
__global__ void __launch_bounds__(kTreeThreads) emat_log_G_tree_kernel(const LogGParams P) {
  __shared__ double s_wsd[kTreeThreads / 32];
  __shared__ int s_wsi[kTreeThreads / 32];
  __shared__ int s_cnt[kMaxPartitions * 4];
  __shared__ int s_ab[16];
  __shared__ double s_carry;
  __shared__ int s_icarry;
  const ForestDev& f = P.f;
  const int tid = threadIdx.x;
  const int tree = blockIdx.x;
  const TreeDev T = f.trees[tree];
  const SitesDev& S = f.sites[T.sites_id];
  if (tid == 0) { s_carry = 0.0; s_icarry = 0; }
  if (tid < 16) s_ab[tid] = 0;
  if (tid < kMaxPartitions * 4) s_cnt[tid] = tid < S.P * 4 ? S.ref_freq[tid] : 0;
  __syncthreads();
  double a1 = 0.0, a2 = 0.0; int m = 0;
  for (int j0 = 0; j0 < T.num_ctiles; j0 += kTreeThreads) {
    const int j = T.first_ctile + j0 + tid;
    const bool ok = j0 + tid < T.num_ctiles;
    const double v = ok ? P.tile_agg[j] : 0.0;
    const int iv = ok ? P.tile_iagg[j] : 0;
    double tot; int itot;
    const double incl = block_scan_incl<double, kTreeThreads>(v, s_wsd, &tot);
    const int iincl = block_scan_incl<int, kTreeThreads>(iv, s_wsi, &itot);
    if (ok) {
      const double pre = s_carry + (incl - v);          // exclusive prefix of this tile
      const int ipre = s_icarry + (iincl - iv);
      P.tile_agg[j] = pre;
      P.tile_iagg[j] = ipre;
      const double A1 = P.tile_part[j * 2 + 0], A2 = P.tile_part[j * 2 + 1];
      a1 += A1 - pre * A2;                              // sum over the tile of -(lambda_local + pre) len + g
      a2 += A2;
      m += P.tile_ipart[j * 17];
    }
    __syncthreads();
    if (tid == 0) { s_carry += tot; s_icarry += itot; }
    __syncthreads();
  }
  // num_muts_ab: 16 bins x tiles, summed by 16-thread groups (integer adds: order irrelevant)
  for (int idx = tid; idx < T.num_ctiles * 16; idx += kTreeThreads) {
    const int c = P.tile_ipart[(size_t)(T.first_ctile + (idx >> 4)) * 17 + 1 + (idx & 15)];
    if (c) atomicAdd(&s_ab[idx & 15], c);
  }
  a1 = block_sum<double, kTreeThreads>(a1, s_wsd);
  a2 = block_sum<double, kTreeThreads>(a2, s_wsd);
  m = block_sum<int, kTreeThreads>(m, s_wsi);
  if (tid == 0) {
    P.tree_out[tree * 4 + 1] = a1;
    P.tree_out[tree * 4 + 2] = a2;
    P.tree_out[tree * 4 + 3] = S.cumQ[S.L] + 0.0;   // (lambda at the root is lambda_out[node_base] after pass 3)
    P.tree_iout[tree * 20 + 0] = m;
    P.tree_iout[tree * 20 + 1] = 0;
  }
  // root prior (core/phylo_tree_calc.cpp:467-504): reference-sequence state counts per partition, adjusted by the
  // root's "mutations", missing sites and from-state overrides.
  {
    const int r = T.node_base;   // the root is the first position of its tree
    for (int i = f.mut_off[r] + tid; i < f.mut_off[r + 1]; i += kTreeThreads) {
      const int code = f.mut_code[i]; const int pt = code >> 4;
      atomicSub(&s_cnt[pt * 4 + ((code >> 2) & 3)], 1);
      atomicAdd(&s_cnt[pt * 4 + (code & 3)], 1);
    }
    for (int i = f.miss_off[r]; i < f.miss_off[r + 1]; ++i) {
      const int2 se = f.miss_se[i]; const int s = se.x, e = se.y;
      for (int l = s + tid; l < e; l += kTreeThreads) atomicSub(&s_cnt[S.part[l] * 4 + S.ref[l]], 1);
    }
    for (int i = f.fs_off[r] + tid; i < f.fs_off[r + 1]; i += kTreeThreads) {
      const int code = f.fs_code[i]; const int pt = code >> 4;
      atomicAdd(&s_cnt[pt * 4 + ((code >> 2) & 3)], 1);
      atomicSub(&s_cnt[pt * 4 + (code & 3)], 1);
    }
  }
  __syncthreads();
  if (tid < 16) P.tree_iout[tree * 20 + 2 + tid] = s_ab[tid];
  if (tid == 0) {
    double lp = 0.0;
    bool impossible = false;
    for (int b = 0; b < S.P; ++b) {
      for (int a = 0; a < 4; ++a) {
        const double pi = S.pi[b * 4 + a];
        const int c = s_cnt[b * 4 + a];
        if (pi != 0.0) lp += c * log(pi);
        else if (c != 0) impossible = true;
      }
    }
    P.tree_out[tree * 4 + 0] = impossible ? -CUDART_INF : lp;
  }
}

// ---- folded fast path (uniform site rates) ------------------------------------------------------------------------------------------------
// With no site-rate heterogeneity every term of a branch's delta-lambda is  mu nu q_a(a)  times an integer that depends only on
// the tree, and so is their sum down the path from the root: ForestDev::C, the per-node state counts built at upload.  lambda_i
// of every node is then one 4P-term dot product, lambda_ref + sum_k mu nu q_a(a) C[q][k], with no dependence between nodes: the
// tile kernel is a streaming pass with no scan and no closer list.  The mutation lists are still walked, in list order, for the
// sum_m [ d_m (t_m - t_P) + log(mu nu q_from,to) ]  part of calc_branch_log_G (core/phylo_tree_calc.h:185-206).  nsmn and the
// num_muts tallies do not depend on the evo model nor on times: they come from the general pass that runs once at upload.
// One CTA per tile of kLgTile positions (the ctile grid of the general schedule), thread tid owning positions tid and
// tid + kLgThreads; the per-tile partials are summed per tree in a fixed order, so log G is bit-reproducible.
// 6 resident CTAs per SM (40 registers, no spills): measured fastest against 4 (64 registers) and 8 (32 registers, with spills)
__global__ void __launch_bounds__(kLgThreads, 6) emat_log_G_folded_kernel(const __grid_constant__ LogGParams P) {
  __shared__ double s_muq[kMaxPartitions * 4];
  __shared__ double s_w[kNW * 2];
  const ForestDev& f = P.f;
  const int tid = threadIdx.x;
  const int tile = blockIdx.x;
  const int4 ct = __ldg(reinterpret_cast<const int4*>(f.ctiles + tile));
  const int tile_start = ct.x, n_act = ct.y;
  const SitesDev& S = f.sites[ct.w];
  const int G = f.fsw_stride / 4;
  if (tid < kMaxPartitions * 4) s_muq[tid] = S.tab_muq[tid];
  const double lambda_ref = __ldg(S.cumQ + S.L);
  __syncthreads();
  double contrib = 0.0, tcontrib = 0.0;
#pragma unroll
  for (int u = 0; u < kLgNPT; ++u) {
    const int q = u * kLgThreads + tid, p = tile_start + q;
    if (q < n_act) {
      const int par = __ldg(f.parent_pos + p);
      const double tN = __ldg(f.t + p);
      const int m0 = __ldg(f.mut_off + p), m1 = __ldg(f.mut_off + p + 1);
      const uint4* c4 = reinterpret_cast<const uint4*>(f.C) + (size_t)p * G;
      double dot = 0.0;
      for (int k = 0; k < G; ++k) {
        const int4 w = __ldg(reinterpret_cast<const int4*>(c4 + k));
        dot += s_muq[4 * k] * (double)w.x + s_muq[4 * k + 1] * (double)w.y + s_muq[4 * k + 2] * (double)w.z + s_muq[4 * k + 3] * (double)w.w;
      }
      const double lam = lambda_ref + dot;
      P.lambda_out[p] = lam;
      if (par >= 0) {        // the root's list ("mutations" above the root) is not part of log G
        const double tP = __ldg(f.t + par);
        double es = 0.0, ds = 0.0;
        for (int i = m0; i < m1; ++i) {
          const int code = __ldg(f.mut_code + i) & 63;
          const double dd = __ldg(S.tab_md + code);
          es += dd * __ldg(f.mut_t + i) + __ldg(S.tab_lq + code);
          ds += dd;
        }
        const double len = tN - tP;
        contrib += -lam * len + (es - tP * ds);
        tcontrib += len;
      }
    }
  }
  const int lane = tid & 31, warp = tid >> 5;
  contrib = warp_sum(contrib); tcontrib = warp_sum(tcontrib);
  if (lane == 0) { s_w[warp * 2 + 0] = contrib; s_w[warp * 2 + 1] = tcontrib; }
  __syncthreads();
  if (warp == 0) {
    double a = lane < kNW ? s_w[lane * 2 + 0] : 0.0;
    double b = lane < kNW ? s_w[lane * 2 + 1] : 0.0;
    a = warp_sum(a); b = warp_sum(b);
    if (lane == 0) { P.tile_part[tile * 2 + 0] = a; P.tile_part[tile * 2 + 1] = b; }
  }
}

// pass 2 of the folded path: one CTA per tree -- the tile partials summed in a fixed order, the tile prefixes of lambda_i set to 0
// (the tile kernel wrote final values; the getter adds the prefix the general schedule leaves there), and the root prior from the
// root's state counts (ref_freq + C[root] is exactly the state count vector of core/phylo_tree_calc.cpp:467-504).
__global__ void __launch_bounds__(kTreeThreads) emat_log_G_folded_tree_kernel(const LogGParams P) {
  __shared__ double s_wsd[kTreeThreads / 32];
  const ForestDev& f = P.f;
  const int tid = threadIdx.x;
  const int tree = blockIdx.x;
  const TreeDev T = f.trees[tree];
  const SitesDev& S = f.sites[T.sites_id];
  double a1 = 0.0, a2 = 0.0;
  for (int j = T.first_ctile + tid; j < T.first_ctile + T.num_ctiles; j += kTreeThreads) {
    a1 += P.tile_part[j * 2 + 0];
    a2 += P.tile_part[j * 2 + 1];
    P.tile_agg[j] = 0.0;
  }
  a1 = block_sum<double, kTreeThreads>(a1, s_wsd);
  a2 = block_sum<double, kTreeThreads>(a2, s_wsd);
  if (tid == 0) {
    P.tree_out[tree * 4 + 1] = a1;
    P.tree_out[tree * 4 + 2] = a2;
    P.tree_out[tree * 4 + 3] = S.cumQ[S.L] + 0.0;
    const int32_t* cr = f.C + (size_t)T.node_base * f.fsw_stride;   // the root is the first position of its tree
    double lp = 0.0;
    bool impossible = false;
    for (int b = 0; b < S.P; ++b) {
      for (int a = 0; a < 4; ++a) {
        const double pi = S.pi[b * 4 + a];
        const int c = S.ref_freq[b * 4 + a] + cr[b * 4 + a];
        if (pi != 0.0) lp += c * log(pi);
        else if (c != 0) impossible = true;
      }
    }
    P.tree_out[tree * 4 + 0] = impossible ? -CUDART_INF : lp;
  }
}

// ---- getters: lambda_i / nsmn are kept on the device as (tile-local value, exclusive prefix of the tile); the two are
// combined when somebody asks for them, in host node order: out[id] = local[pos] + prefix[tile(pos)].
template <typename V>
__global__ void gather_host_order_kernel(const int32_t* __restrict__ pos_of_node, const V* __restrict__ src, const V* __restrict__ tile_prefix,
                                         V* __restrict__ dst, int node_base, int first_ctile, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const int pos = pos_of_node[node_base + i];
    dst[i] = src[node_base + pos] + tile_prefix[first_ctile + pos / kLgTile];
  }
}

int gather_lambda_host_order(dphy_ctx* ctx, dphy_forest* fo, int tree, double* d_dst) {
  const TreeDev& T = fo->trees[tree];
  gather_host_order_kernel<double><<<(T.num_nodes + 255) / 256, 256, 0, ctx->stream>>>(fo->h.pos_of_node, fo->d_lambda, fo->d_tile_agg, d_dst,
                                                                                       T.node_base, T.first_ctile, T.num_nodes);
  ctx->launches += 1;
  return check_cuda(ctx, cudaGetLastError(), "gather_host_order_kernel<double>");
}
int gather_nsmn_host_order(dphy_ctx* ctx, dphy_forest* fo, int tree, int32_t* d_dst) {
  const TreeDev& T = fo->trees[tree];
  gather_host_order_kernel<int32_t><<<(T.num_nodes + 255) / 256, 256, 0, ctx->stream>>>(fo->h.pos_of_node, fo->d_nsmn, fo->d_tile_iagg, d_dst,
                                                                                        T.node_base, T.first_ctile, T.num_nodes);
  ctx->launches += 1;
  return check_cuda(ctx, cudaGetLastError(), "gather_host_order_kernel<int>");
}

int launch_log_G_general(dphy_ctx* ctx, dphy_forest* fo) {
  if (fo->h.num_ctiles == 0) return DPHY_OK;
  int st = refresh_sites(ctx, fo);
  if (st != DPHY_OK) return st;
  LogGParams P;
  P.f = fo->h;
  P.lambda_out = fo->d_lambda;
  P.nsmn_out = fo->d_nsmn;
  P.tile_agg = fo->d_tile_agg;
  P.tile_iagg = fo->d_tile_iagg;
  P.tile_part = fo->d_tile_part;
  P.tile_ipart = fo->d_tile_ipart;
  P.tree_out = fo->d_tree_out;
  P.tree_iout = fo->d_tree_iout;
  P.sd_delta = fo->d_sd_delta;
  P.sd_n = fo->d_sd_n;
  P.strad_list = fo->d_strad_list;
  P.num_strad = fo->num_strad;
  if (P.num_strad > 0) {
    emat_log_G_straddler_kernel<<<(P.num_strad + 127) / 128, 128, 0, ctx->stream>>>(P);
    ctx->launches += 1;
  }
  // The direct-from-global tile kernel: every thread walks the short lists of its own two nodes.  (A TMA-staged persistent variant
  // -- node records / event lists / closer slice brought to shared memory by cp.async.bulk under an mbarrier, two stages deep -- was
  // built and measured in round 1: 281 vs 216 us per 16 x 100k-tip evaluation.  With ~2 events per node, 8 resident CTAs/SM walking
  // lists keep more loads in flight than two staged tiles per SM; it was removed.)  Tiles go in fo->d_ctile_order: full tiles
  // first, the partly filled ones last.
  emat_log_G_tile_kernel<<<fo->h.num_ctiles, kLgThreads, 0, ctx->stream>>>(P, fo->d_ctile_order);
  ctx->launches += 1;
  emat_log_G_tree_kernel<<<fo->h.num_trees, kTreeThreads, 0, ctx->stream>>>(P);
  ctx->launches += 1;
  st = check_cuda(ctx, cudaGetLastError(), "emat_log_G kernels launch");
  if (st == DPHY_OK) fo->struct_valid = true;
  return st;
}

static int launch_log_G_folded(dphy_ctx* ctx, dphy_forest* fo) {
  int st = refresh_sites(ctx, fo);
  if (st != DPHY_OK) return st;
  LogGParams P{};
  P.f = fo->h;
  P.lambda_out = fo->d_lambda;
  P.tile_agg = fo->d_tile_agg;
  P.tile_part = fo->d_tile_part;
  P.tree_out = fo->d_tree_out;
  const int grid = fo->h.num_ctiles;
  // profiling only: DPHY_FOLDED_REPEAT=n launches the tile kernel n times per evaluation (idempotent), to separate its in-stream
  // duration from launch gaps and the per-tree kernel
  static const int repeat = [] { const char* e = getenv("DPHY_FOLDED_REPEAT"); return e ? std::max(1, atoi(e)) : 1; }();
  for (int rep = 0; rep < repeat; ++rep) emat_log_G_folded_kernel<<<grid, kLgThreads, 0, ctx->stream>>>(P);
  // one CTA per tree folds the tile partials (fusing this into the tile kernel with a last-CTA ticket was measured slower:
  // every CTA then waits a device-wide atomic round trip before it can retire -- 102 vs 96 us per evaluation)
  emat_log_G_folded_tree_kernel<<<fo->h.num_trees, kTreeThreads, 0, ctx->stream>>>(P);
  ctx->launches += 2;
  return check_cuda(ctx, cudaGetLastError(), "emat_log_G folded kernels launch");
}

int launch_log_G(dphy_ctx* ctx, dphy_forest* fo) {
  if (fo->h.num_ctiles == 0) return DPHY_OK;
  bool all_uniform = true;
  for (const dphy_sites* s : fo->sites) all_uniform = all_uniform && s->h.nu_uniform;
  // the folded path leaves nsmn and the num_muts tallies alone: the getters that return those run a general pass on demand
  // (fo->struct_valid says whether one has run since the upload)
  if (ctx->logg_path == 0 && all_uniform) return launch_log_G_folded(ctx, fo);
  return launch_log_G_general(ctx, fo);
}

}  // namespace dphy
