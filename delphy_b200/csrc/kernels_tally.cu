// kernels_tally.cu -- per-tree tallies that feed the reference's global (Gibbs) moves (sm_100a).
//
//   calc_num_muts_beta_ab   core/phylo_tree_calc.cpp:599-610   (int, bit-exact)
//   calc_num_muts_l         core/phylo_tree_calc.cpp:612-622   (int, bit-exact)
//   calc_num_muts_l_ab      core/phylo_tree_calc.cpp:624-634   (int, bit-exact)
//   calc_Ttwiddle_beta_a    core/phylo_tree_calc.cpp:288-369   (fp64)
//   calc_Ttwiddle_l         core/phylo_tree_calc.cpp:176-222   (fp64)
//   calc_T_l_a              core/phylo_tree_calc.cpp:130-174   (fp64)
//
// The reference's Ttwiddle_beta_a walks the tree carrying the 4P-vector ntwiddle and loops over EVERY missing site
// of every missation interval.  Here all three time tallies use the "total branch length below" form the reference
// itself uses for calc_T_l_a: in DFS pre-order the subtree of p is the contiguous range [p, p+size), so
// T_below(p) = PL[p+size-1] - PL[p] with PL the inclusive scan of branch lengths -- one plain scan -- and every
// mutation / interval / from-state override becomes an independent term.  Per-site interval loops are replaced by
// look-ups in cumulative tables (cum_nu_ba for Ttwiddle_beta_a; a +-T difference array scanned once for the
// per-site outputs).
#include "dphy_internal.h"
#include "device_utils.cuh"

#include <algorithm>
#include <cstring>
#include <optional>

namespace dphy {

// ---- inclusive scan of branch lengths over one tree's device positions --------------------------------------------
// Same single-pass scheme as the log-G kernel: tile aggregate published with a release flag, predecessors of the
// same tree summed in a fixed order.
__global__ void __launch_bounds__(kTile) tally_branch_len_scan_kernel(ForestDev f, int tree, double* __restrict__ PL,
                                                                      double* tile_agg, uint32_t* tile_flag,
                                                                      uint32_t* ticket, uint32_t epoch) {
  __shared__ double s_ws[kTile / 32];
  __shared__ double s_prefix;
  __shared__ int s_tile;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_tile = (int)atomicAdd(ticket, 1u);
  __syncthreads();
  const int tile = s_tile;
  const TreeDev T = f.trees[tree];
  const int p = T.node_base + tile * kTile + tid;
  double len = 0.0;
  if (p < T.node_base + T.num_nodes) {
    const int par = f.parent_pos[p];
    if (par >= 0) len = f.t[p] - f.t[par];
  }
  double tot;
  const double incl = block_scan_incl<double, kTile>(len, s_ws, &tot);
  if (tid == 0) {
    tile_agg[tile] = tot;
    __threadfence();
    st_release_u32(tile_flag + tile, epoch);
    if (tile == T.num_tiles - 1) ticket[0] = 0u;   // every ticket has been handed out: re-arm
  }
  if (warp == 0) {
    double acc = 0.0;
    for (int j0 = 0; j0 < tile; j0 += 32) {
      const int j = j0 + lane;
      if (j < tile) {
        while (ld_acquire_u32(tile_flag + j) != epoch) { __nanosleep(20); }
        acc += ld_cg_f64(tile_agg + j);
      }
    }
    acc = warp_sum(acc);
    if (lane == 0) s_prefix = acc;
  }
  __syncthreads();
  if (p < T.node_base + T.num_nodes) PL[p - T.node_base] = s_prefix + incl;
}

// Order-independent fp64 accumulation.  The per-site tallies scatter ~(M + I + F) terms into L bins from all over the tree; fp64
// atomicAdd would make the sums depend on the arrival order (not reproducible run to run, which a replayed Gibbs move would see).
// Each term is split into its integer part and its fraction rounded to 2^-44, and both are accumulated with INTEGER atomics, which
// commute exactly: the result is the exact sum of the rounded terms, whatever the order.  Error <= 2^-45 (3e-14, absolute) per term.
__device__ __forceinline__ void fx_add(long long* __restrict__ acc2, double v) {
  const double hi = trunc(v);
  const long long ih = (long long)hi;
  const long long il = __double2ll_rn((v - hi) * 17592186044416.0);        // 2^44
  if (ih) atomicAdd(reinterpret_cast<unsigned long long*>(acc2), (unsigned long long)ih);
  if (il) atomicAdd(reinterpret_cast<unsigned long long*>(acc2 + 1), (unsigned long long)il);
}
__device__ __forceinline__ double fx_get(const long long* __restrict__ acc2) {
  return (double)acc2[0] + (double)acc2[1] * 5.6843418860808015e-14;        // 2^-44
}
// the lanes of a warp that hit the same bin combine first (interval end points pile up on a few sites: every tip's 5' / 3' end gap
// starts at site 0 / ends at site L, and same-address atomics serialise in L2); ascending lanes, so the partial sum is reproducible
__device__ __forceinline__ void warp_agg_fx_add(long long* base2, int idx, double v) {
  const unsigned peers = __match_any_sync(__activemask(), idx);
  double sum = 0.0;
  for (unsigned rem = peers; rem; rem &= rem - 1) sum += __shfl_sync(peers, v, __ffs(rem) - 1);
  if ((int)(threadIdx.x & 31) == __ffs(peers) - 1) fx_add(base2 + 2 * (size_t)idx, sum);
}

struct TallyOut {
  int32_t* num_muts_beta_ab;  // [P*16] or null
  int32_t* num_muts_l;        // [L] or null
  int32_t* num_muts_l_ab;     // [L*16] or null
  double* beta_a_part;        // [num_tiles * 16] per-tile partials of Ttwiddle_beta_a, or null
  long long* Ttw_l;           // [L][2] fixed-point accumulators (fx_add) or null
  long long* T_l_a;           // [L*4][2] or null
  long long* miss_diff;       // [L+1][2] difference array of T_below_miss (needed when Ttw_l or T_l_a)
};

// One thread per node of the tree.  kTime: evaluate the time tallies (needs PL).
template <bool kTime>
__global__ void __launch_bounds__(kTile) tally_events_kernel(ForestDev f, int tree, const double* __restrict__ PL,
                                                             const double* __restrict__ cum_nu_ba, TallyOut out) {
  __shared__ int s_bab[kMaxPartitions * 16];
  __shared__ double s_ws[kTile / 32];
  const int tid = threadIdx.x;
  const TreeDev T = f.trees[tree];
  const SitesDev& S = f.sites[T.sites_id];
  const int L = S.L, P = S.P;
  if (tid < kMaxPartitions * 16) s_bab[tid] = 0;
  __syncthreads();
  const int q = blockIdx.x * kTile + tid;
  const int p = T.node_base + q;
  const bool active = q < T.num_nodes;
  double acc[kMaxPartitions * 4];
#pragma unroll
  for (int k = 0; k < kMaxPartitions * 4; ++k) acc[k] = 0.0;

  if (active) {
    const int par = f.parent_pos[p];
    const bool is_root = par < 0;
    double Tb = 0.0, len = 0.0, tN = 0.0;
    if (kTime) {
      const int last = q + f.subtree_size[p] - 1;
      Tb = PL[last] - PL[q];
      tN = f.t[p];
      len = is_root ? 0.0 : tN - f.t[par];
    }
    for (int i = f.mut_off[p]; i < f.mut_off[p + 1]; ++i) {
      const int l = f.mut_site[i], code = f.mut_code[i], ft = code & 15, from = ft >> 2, to = ft & 3;
      const int pt = code >> 4;
      if (!is_root) {   // "mutations" above the root are just deltas from the reference sequence
        if (out.num_muts_beta_ab) atomicAdd(&s_bab[pt * 16 + ft], 1);
        if (out.num_muts_l) atomicAdd(out.num_muts_l + l, 1);
        if (out.num_muts_l_ab) atomicAdd(out.num_muts_l_ab + (size_t)l * 16 + ft, 1);
      }
      if (kTime) {
        const double Tbm = Tb + (is_root ? 0.0 : tN - f.mut_t[i]);
        if (out.beta_a_part) {
          const double w = S.nu[l] * Tbm;
#pragma unroll
          for (int k = 0; k < kMaxPartitions * 4; ++k) {
            if (k == pt * 4 + from) acc[k] -= w;
            if (k == pt * 4 + to) acc[k] += w;
          }
        }
        if (out.Ttw_l) fx_add(out.Ttw_l + 2 * (size_t)l, ((-S.q[pt * 16 + to * 5]) - (-S.q[pt * 16 + from * 5])) * Tbm);
        if (out.T_l_a) { fx_add(out.T_l_a + 2 * ((size_t)l * 4 + from), -Tbm); fx_add(out.T_l_a + 2 * ((size_t)l * 4 + to), Tbm); }
      }
    }
    if (kTime) {
      const double Tbmiss = Tb + len;
      for (int i = f.miss_off[p]; i < f.miss_off[p + 1]; ++i) {
        const int2 se = f.miss_se[i]; const int s = se.x, e = se.y;
        if (out.beta_a_part) {
#pragma unroll
          for (int k = 0; k < kMaxPartitions * 4; ++k) {
            if (k < P * 4) {
              const double* c = cum_nu_ba + (size_t)k * (L + 1);
              acc[k] -= (c[e] - c[s]) * Tbmiss;
            }
          }
        }
        if (out.miss_diff) { warp_agg_fx_add(out.miss_diff, s, Tbmiss); warp_agg_fx_add(out.miss_diff, e, -Tbmiss); }
      }
      for (int i = f.fs_off[p]; i < f.fs_off[p + 1]; ++i) {
        const int l = f.fs_site[i], code = f.fs_code[i], from = code & 3, rf = (code >> 2) & 3, pt = code >> 4;
        if (out.beta_a_part) {
          const double w = S.nu[l] * Tbmiss;
#pragma unroll
          for (int k = 0; k < kMaxPartitions * 4; ++k) {
            if (k == pt * 4 + rf) acc[k] += w;      // undo the ref-seq assumption
            if (k == pt * 4 + from) acc[k] -= w;    // apply the correct from-state
          }
        }
        if (out.Ttw_l) fx_add(out.Ttw_l + 2 * (size_t)l, ((-S.q[pt * 16 + rf * 5]) - (-S.q[pt * 16 + from * 5])) * Tbmiss);
        if (out.T_l_a) { fx_add(out.T_l_a + 2 * ((size_t)l * 4 + rf), Tbmiss); fx_add(out.T_l_a + 2 * ((size_t)l * 4 + from), -Tbmiss); }
      }
    }
  }
  if (kTime && out.beta_a_part) {
#pragma unroll
    for (int k = 0; k < kMaxPartitions * 4; ++k) {
      const double v = block_sum<double, kTile>(acc[k], s_ws);
      if (tid == 0) out.beta_a_part[(size_t)blockIdx.x * 16 + k] = v;
    }
  }
  __syncthreads();
  if (out.num_muts_beta_ab && tid < P * 16 && s_bab[tid] != 0) atomicAdd(out.num_muts_beta_ab + tid, s_bab[tid]);
}

// Ttwiddle_beta_a = ntwiddle_ref * T_total + sum over tiles (fixed order).
__global__ void tally_beta_a_finalize_kernel(ForestDev f, int tree, const double* __restrict__ PL,
                                             const double* __restrict__ cum_nu_ba, const double* __restrict__ part,
                                             int num_tiles, double* __restrict__ out) {
  const TreeDev T = f.trees[tree];
  const SitesDev& S = f.sites[T.sites_id];
  const int k = threadIdx.x;
  if (k >= S.P * 4) return;
  const double Ttot = PL[T.num_nodes - 1];
  double v = cum_nu_ba[(size_t)k * (S.L + 1) + S.L] * Ttot;
  for (int j = 0; j < num_tiles; ++j) v += part[(size_t)j * 16 + k];
  out[k] = v;
}

// Per-site finalize: scan the +-T_below_miss difference array over sites, then add the no-mutation baseline
// (T_total - missing time) * [state == ref].  One CTA sweeping coalesced slabs with a running carry (L is at most a few 1e5).
__global__ void __launch_bounds__(1024) tally_sites_finalize_kernel(ForestDev f, int tree, const double* __restrict__ PL,
                                                                    const long long* __restrict__ miss_diff,
                                                                    const long long* __restrict__ Ttw_fx, const long long* __restrict__ T_l_a_fx,
                                                                    double* __restrict__ Ttw_l, double* __restrict__ T_l_a) {
  __shared__ double s_ws[32];
  __shared__ double s_carry;
  const TreeDev T = f.trees[tree];
  const SitesDev& S = f.sites[T.sites_id];
  const int L = S.L, tid = threadIdx.x;
  const double Ttot = PL[T.num_nodes - 1];
  if (tid == 0) s_carry = 0.0;
  __syncthreads();
  // slabs of 4,096 sites, 4 consecutive sites per thread: every load / store of a warp is one contiguous run
  constexpr int kPer = 4;
  for (int base = 0; base < L; base += 1024 * kPer) {
    const int l0 = base + tid * kPer;
    double v[kPer], tot = 0.0;
#pragma unroll
    for (int u = 0; u < kPer; ++u) { v[u] = l0 + u < L ? fx_get(miss_diff + 2 * (size_t)(l0 + u)) : 0.0; tot += v[u]; }
    double bt;
    const double incl = block_scan_incl<double, 1024>(tot, s_ws, &bt);
    double run = s_carry + (incl - tot);
#pragma unroll
    for (int u = 0; u < kPer; ++u) {
      const int l = l0 + u;
      run += v[u];
      if (l < L) {
        const double basev = Ttot - run;    // time during which site l is present with the reference state (before mutations)
        const int a = S.ref[l], pt = S.part[l];
        if (Ttw_l) Ttw_l[l] = fx_get(Ttw_fx + 2 * (size_t)l) + (-S.q[pt * 16 + a * 5]) * basev;
        if (T_l_a) {
#pragma unroll
          for (int b = 0; b < 4; ++b) T_l_a[(size_t)l * 4 + b] = fx_get(T_l_a_fx + 2 * ((size_t)l * 4 + b)) + (b == a ? basev : 0.0);
        }
      }
    }
    __syncthreads();
    if (tid == 0) s_carry += bt;
    __syncthreads();
  }
}

// ---- host-side launchers -------------------------------------------------------------------------------------------
static int scan_branch_lengths(dphy_ctx* ctx, dphy_forest* fo, int tree, double** PL_out) {
  const TreeDev& T = fo->trees[tree];
  double* PL = (double*)ctx->arena.alloc(sizeof(double) * T.num_nodes);
  // own scan workspace: d_tile_agg holds the log-G tile prefixes that the lambda_i getter still needs
  double* agg = (double*)ctx->arena.alloc(sizeof(double) * T.num_tiles);
  // ... and its own tile ticket: the trees of a forest are scanned side by side on several streams (dphy_forest_calc_site_tallies),
  // and a ticket shared by two running scans would hand one tree's tiles to the other -- its CTAs would wait for ever
  uint32_t* ticket = (uint32_t*)ctx->arena.alloc(sizeof(uint32_t));
  if (!PL || !agg || !ticket) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "arena exhausted (tally PL)");
  DPHY_CUDA(ctx, cudaMemsetAsync(ticket, 0, sizeof(uint32_t), ctx->stream));
  fo->epoch += 1; if (fo->epoch == 0) fo->epoch = 1;
  tally_branch_len_scan_kernel<<<T.num_tiles, kTile, 0, ctx->stream>>>(fo->h, tree, PL, agg,
                                                                       fo->d_tile_flag + T.first_tile, ticket, fo->epoch);
  ctx->launches += 1;
  *PL_out = PL;
  return check_cuda(ctx, cudaGetLastError(), "tally_branch_len_scan_kernel");
}

// defer: leave the device->host copies enqueued and the arena scope open; the caller synchronizes the stream and releases the
// arena once for a whole batch of trees (dphy_forest_calc_site_tallies)
int tally_num_muts(dphy_ctx* ctx, dphy_forest* fo, int tree, int32_t* out_beta_ab, int32_t* out_l, int32_t* out_l_ab, bool defer = false) {
  const TreeDev& T = fo->trees[tree];
  const dphy_sites* s = fo->sites[T.sites_id];
  int st = refresh_sites(ctx, fo);
  if (st != DPHY_OK) return st;
  const size_t mark = ctx->arena.mark();
  const int L = s->L, P = s->P;
  TallyOut o{};
  if (out_beta_ab) o.num_muts_beta_ab = (int32_t*)ctx->arena.alloc(sizeof(int32_t) * P * 16);
  if (out_l) o.num_muts_l = (int32_t*)ctx->arena.alloc(sizeof(int32_t) * L);
  if (out_l_ab) o.num_muts_l_ab = (int32_t*)ctx->arena.alloc(sizeof(int32_t) * (size_t)L * 16);
  if ((out_beta_ab && !o.num_muts_beta_ab) || (out_l && !o.num_muts_l) || (out_l_ab && !o.num_muts_l_ab)) {
    ctx->arena.release(mark);
    return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "arena exhausted (num_muts tallies)");
  }
  if (o.num_muts_beta_ab) DPHY_CUDA(ctx, cudaMemsetAsync(o.num_muts_beta_ab, 0, sizeof(int32_t) * P * 16, ctx->stream));
  if (o.num_muts_l) DPHY_CUDA(ctx, cudaMemsetAsync(o.num_muts_l, 0, sizeof(int32_t) * L, ctx->stream));
  if (o.num_muts_l_ab) DPHY_CUDA(ctx, cudaMemsetAsync(o.num_muts_l_ab, 0, sizeof(int32_t) * (size_t)L * 16, ctx->stream));
  tally_events_kernel<false><<<T.num_tiles, kTile, 0, ctx->stream>>>(fo->h, tree, nullptr, nullptr, o);
  ctx->launches += 1;
  st = check_cuda(ctx, cudaGetLastError(), "tally_events_kernel<false>");
  if (st == DPHY_OK && out_beta_ab) st = check_cuda(ctx, cudaMemcpyAsync(out_beta_ab, o.num_muts_beta_ab, sizeof(int32_t) * P * 16, cudaMemcpyDeviceToHost, ctx->stream), "D2H");
  if (st == DPHY_OK && out_l && defer) ctx->deferred_d2h.push_back({out_l, o.num_muts_l, sizeof(int32_t) * (size_t)L});
  else if (st == DPHY_OK && out_l) st = check_cuda(ctx, cudaMemcpyAsync(out_l, o.num_muts_l, sizeof(int32_t) * L, cudaMemcpyDeviceToHost, ctx->stream), "D2H");
  if (st == DPHY_OK && out_l_ab) st = check_cuda(ctx, cudaMemcpyAsync(out_l_ab, o.num_muts_l_ab, sizeof(int32_t) * (size_t)L * 16, cudaMemcpyDeviceToHost, ctx->stream), "D2H");
  if (defer && st == DPHY_OK) return st;
  if (st == DPHY_OK) st = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "num_muts tallies");
  ctx->arena.release(mark);
  return st;
}

int tally_times(dphy_ctx* ctx, dphy_forest* fo, int tree, double* out_beta_a, double* out_l, double* out_l_a, bool defer = false) {
  const TreeDev& T = fo->trees[tree];
  const dphy_sites* s = fo->sites[T.sites_id];
  int st = refresh_sites(ctx, fo);
  if (st != DPHY_OK) return st;
  const size_t mark = ctx->arena.mark();
  const int L = s->L, P = s->P;
  double* PL = nullptr;
  st = scan_branch_lengths(ctx, fo, tree, &PL);
  if (st != DPHY_OK) { ctx->arena.release(mark); return st; }
  TallyOut o{};
  double* d_beta_a = nullptr;
  double* d_Ttw = nullptr; double* d_Tla = nullptr;      // the doubles handed back (the scatter itself runs on fixed-point bins)
  if (out_beta_a) {
    o.beta_a_part = (double*)ctx->arena.alloc(sizeof(double) * 16 * T.num_tiles);
    d_beta_a = (double*)ctx->arena.alloc(sizeof(double) * 16);
  }
  if (out_l) { o.Ttw_l = (long long*)ctx->arena.alloc(sizeof(long long) * 2 * L); d_Ttw = (double*)ctx->arena.alloc(sizeof(double) * L); }
  if (out_l_a) { o.T_l_a = (long long*)ctx->arena.alloc(sizeof(long long) * 2 * (size_t)L * 4); d_Tla = (double*)ctx->arena.alloc(sizeof(double) * (size_t)L * 4); }
  if (out_l || out_l_a) o.miss_diff = (long long*)ctx->arena.alloc(sizeof(long long) * 2 * (L + 1));
  if ((out_beta_a && (!o.beta_a_part || !d_beta_a)) || (out_l && (!o.Ttw_l || !d_Ttw)) || (out_l_a && (!o.T_l_a || !d_Tla)) || ((out_l || out_l_a) && !o.miss_diff)) {
    ctx->arena.release(mark);
    return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "arena exhausted (time tallies)");
  }
  if (o.Ttw_l) DPHY_CUDA(ctx, cudaMemsetAsync(o.Ttw_l, 0, sizeof(long long) * 2 * L, ctx->stream));
  if (o.T_l_a) DPHY_CUDA(ctx, cudaMemsetAsync(o.T_l_a, 0, sizeof(long long) * 2 * (size_t)L * 4, ctx->stream));
  if (o.miss_diff) DPHY_CUDA(ctx, cudaMemsetAsync(o.miss_diff, 0, sizeof(long long) * 2 * (L + 1), ctx->stream));
  tally_events_kernel<true><<<T.num_tiles, kTile, 0, ctx->stream>>>(fo->h, tree, PL, s->d_cum_nu_ba, o);
  ctx->launches += 1;
  st = check_cuda(ctx, cudaGetLastError(), "tally_events_kernel<true>");
  if (st == DPHY_OK && out_beta_a) {
    tally_beta_a_finalize_kernel<<<1, 32, 0, ctx->stream>>>(fo->h, tree, PL, s->d_cum_nu_ba, o.beta_a_part, T.num_tiles, d_beta_a);
    ctx->launches += 1;
    st = check_cuda(ctx, cudaGetLastError(), "tally_beta_a_finalize_kernel");
    if (st == DPHY_OK) st = check_cuda(ctx, cudaMemcpyAsync(out_beta_a, d_beta_a, sizeof(double) * P * 4, cudaMemcpyDeviceToHost, ctx->stream), "D2H");
  }
  if (st == DPHY_OK && (out_l || out_l_a)) {
    tally_sites_finalize_kernel<<<1, 1024, 0, ctx->stream>>>(fo->h, tree, PL, o.miss_diff, o.Ttw_l, o.T_l_a, d_Ttw, d_Tla);
    ctx->launches += 1;
    st = check_cuda(ctx, cudaGetLastError(), "tally_sites_finalize_kernel");
    if (st == DPHY_OK && out_l && defer) ctx->deferred_d2h.push_back({out_l, d_Ttw, sizeof(double) * (size_t)L});
    else if (st == DPHY_OK && out_l) st = check_cuda(ctx, cudaMemcpyAsync(out_l, d_Ttw, sizeof(double) * L, cudaMemcpyDeviceToHost, ctx->stream), "D2H");
    if (st == DPHY_OK && out_l_a) st = check_cuda(ctx, cudaMemcpyAsync(out_l_a, d_Tla, sizeof(double) * (size_t)L * 4, cudaMemcpyDeviceToHost, ctx->stream), "D2H");
  }
  if (defer && st == DPHY_OK) return st;
  if (st == DPHY_OK) st = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "time tallies");
  ctx->arena.release(mark);
  return st;
}

// Sum over the trees of a forest (fixed order) of the additive per-cycle quantities, packed as doubles for ONE all-reduce:
//   out[0] = sum log_G, [1] = sum T, [2] = sum num_muts, [3..19) = sum num_muts_ab, [19 .. 19 + 4 maxP) = sum Ttwiddle_beta_a
__global__ void pack_cycle_tallies_kernel(ForestDev f, const double* __restrict__ tree_out, const int32_t* __restrict__ tree_iout,
                                          const double* __restrict__ beta_a /* [num_trees][16] */, int maxP4, double* __restrict__ out) {
  const int k = threadIdx.x;
  if (k >= 19 + maxP4) return;
  double v = 0.0;
  for (int t = 0; t < f.num_trees; ++t) {
    if (k == 0) v += (f.trees[t].includes_run_root ? tree_out[t * 4 + 0] : 0.0) + tree_out[t * 4 + 1];
    else if (k == 1) v += tree_out[t * 4 + 2];
    else if (k == 2) v += (double)tree_iout[t * 20 + 0];
    else if (k < 19) v += (double)tree_iout[t * 20 + 2 + (k - 3)];
    else if (k - 19 < f.sites[f.trees[t].sites_id].P * 4) v += beta_a[t * 16 + (k - 19)];
  }
  out[k] = v;
}

}  // namespace dphy

using namespace dphy;

extern "C" {

int dphy_forest_cycle_tallies_device(dphy_ctx* ctx, dphy_forest* fo, double* d_out, int32_t cap) {
  if (!ctx || !fo || !d_out) return DPHY_ERR_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  int maxP = 1;
  for (const dphy_sites* s : fo->sites) maxP = std::max(maxP, (int)s->P);
  if (cap < 19 + 4 * maxP) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "cycle tallies: output shorter than 19 + 4 P doubles");
  int st = refresh_sites(ctx, fo);
  if (st != DPHY_OK) return st;
  // log G under the current model + the structure-only counts (general schedule once per upload)
  if (!fo->struct_valid) st = launch_log_G_general(ctx, fo);
  else if (!fo->eval_current()) st = launch_log_G(ctx, fo);
  if (st != DPHY_OK) return st;
  fo->evaluated = true;
  fo->eval_version.resize(fo->sites.size());
  for (size_t i = 0; i < fo->sites.size(); ++i) fo->eval_version[i] = fo->sites[i]->version;
  const size_t mark = ctx->arena.mark();
  const int nt = fo->h.num_trees;
  double* d_beta = (double*)ctx->arena.alloc(sizeof(double) * 16 * (size_t)std::max(nt, 1));
  if (!d_beta) { ctx->arena.release(mark); return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "arena exhausted (cycle tallies)"); }
  for (int k = 0; k < nt && st == DPHY_OK; ++k) {
    const TreeDev& T = fo->trees[k];
    const dphy_sites* s = fo->sites[T.sites_id];
    double* PL = nullptr;
    st = scan_branch_lengths(ctx, fo, k, &PL);
    if (st != DPHY_OK) break;
    TallyOut o{};
    o.beta_a_part = (double*)ctx->arena.alloc(sizeof(double) * 16 * T.num_tiles);
    if (!o.beta_a_part) { st = set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "arena exhausted (cycle tallies)"); break; }
    tally_events_kernel<true><<<T.num_tiles, kTile, 0, ctx->stream>>>(fo->h, k, PL, s->d_cum_nu_ba, o);
    tally_beta_a_finalize_kernel<<<1, 32, 0, ctx->stream>>>(fo->h, k, PL, s->d_cum_nu_ba, o.beta_a_part, T.num_tiles, d_beta + 16 * (size_t)k);
    ctx->launches += 2;
  }
  if (st == DPHY_OK) {
    pack_cycle_tallies_kernel<<<1, 64, 0, ctx->stream>>>(fo->h, fo->d_tree_out, fo->d_tree_iout, d_beta, 4 * maxP, d_out);
    ctx->launches += 1;
    st = check_cuda(ctx, cudaGetLastError(), "cycle tallies kernels");
  }
  // stream-ordered: the arena scope is reused only by later work on the same stream
  ctx->arena.release(mark);
  return st;
}

int dphy_forest_calc_num_muts_beta_ab(dphy_ctx* ctx, dphy_forest* fo, int32_t tree, int32_t* out) {
  if (!ctx || !fo || !out || tree < 0 || tree >= fo->h.num_trees) return DPHY_ERR_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  return tally_num_muts(ctx, fo, tree, out, nullptr, nullptr);
}

int dphy_forest_calc_num_muts_l(dphy_ctx* ctx, dphy_forest* fo, int32_t tree, int32_t* out_l, int32_t* out_l_ab) {
  if (!ctx || !fo || (!out_l && !out_l_ab) || tree < 0 || tree >= fo->h.num_trees) return DPHY_ERR_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  return tally_num_muts(ctx, fo, tree, nullptr, out_l, out_l_ab);
}

int dphy_forest_calc_Ttwiddle_beta_a(dphy_ctx* ctx, dphy_forest* fo, int32_t tree, double* out) {
  if (!ctx || !fo || !out || tree < 0 || tree >= fo->h.num_trees) return DPHY_ERR_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  return tally_times(ctx, fo, tree, out, nullptr, nullptr);
}

int dphy_forest_calc_site_tallies(dphy_ctx* ctx, dphy_forest* fo, int64_t ld, double* out_Ttwiddle_l, int32_t* out_num_muts_l) {
  if (!ctx || !fo || (!out_Ttwiddle_l && !out_num_muts_l) || ld <= 0) return DPHY_ERR_INVALID_ARGUMENT;
  for (const TreeDev& T : fo->trees)
    if (fo->sites[T.sites_id]->L > ld) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "site tallies: row stride smaller than a tree's number of sites");
  cudaSetDevice(ctx->device);
  const size_t mark = ctx->arena.mark();
  int st = DPHY_OK;
  ctx->deferred_d2h.clear();
  // a device->host copy into pageable memory blocks the host, so the copies are issued after every tree's kernels are enqueued
  // the results come back through the ctx's pinned slab in one go (a device->host copy straight into pageable memory blocks the
  // host for every row), then are copied out to the caller's rows
  auto drain = [&]() {
    size_t total = 0;
    for (const auto& c : ctx->deferred_d2h) total += align_up(c.bytes);
    std::optional<PinnedStage> pin;
    if (total) pin.emplace(ctx, total);
    int r = pin ? pin->status : DPHY_OK;
    char* hb = pin ? pin->p : nullptr;
    size_t off = 0;
    for (const auto& c : ctx->deferred_d2h) {
      if (r == DPHY_OK) r = check_cuda(ctx, cudaMemcpyAsync(hb + off, c.src, c.bytes, cudaMemcpyDeviceToHost, ctx->stream), "site tallies D2H");
      off += align_up(c.bytes);
    }
    const int r2 = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "site tallies");
    if (r == DPHY_OK && r2 == DPHY_OK) {
      off = 0;
      for (const auto& c : ctx->deferred_d2h) { std::memcpy(c.dst, hb + off, c.bytes); off += align_up(c.bytes); }
    }
    ctx->deferred_d2h.clear();
    ctx->arena.release(mark);
    return r != DPHY_OK ? r : r2;
  };
  // Every tree's kernels are enqueued back to back, tree k on side stream k % 4: a tree's sequence is a branch-length scan, an
  // atomics-bound scatter and a one-CTA per-site finalize, none of which fills the GPU, so four trees run side by side (fork after
  // what the main stream holds so far, join before the results are copied back).  One synchronization per arena-full of trees.
  constexpr int kS = dphy_ctx::kTallyStreams;
  cudaStream_t main_stream = ctx->stream;
  bool forked = false;
  if (fo->h.num_trees > 1) {
    bool ok = true;
    for (int i = 0; i < kS && ok; ++i) {
      if (!ctx->tally_streams[i]) ok = cudaStreamCreateWithFlags(&ctx->tally_streams[i], cudaStreamNonBlocking) == cudaSuccess &&
                                       cudaEventCreateWithFlags(&ctx->ev_tally[i], cudaEventDisableTiming) == cudaSuccess;
    }
    if (ok && !ctx->ev_fork) ok = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) == cudaSuccess;
    if (ok) {
      st = refresh_sites(ctx, fo);                      // (on the main stream, before the fork; the per-tree calls then find it done)
      cudaEventRecord(ctx->ev_fork, main_stream);
      for (int i = 0; i < kS; ++i) cudaStreamWaitEvent(ctx->tally_streams[i], ctx->ev_fork, 0);
      forked = true;
    } else cudaGetLastError();
  }
  auto join = [&]() {
    if (!forked) return;
    for (int i = 0; i < kS; ++i) { cudaEventRecord(ctx->ev_tally[i], ctx->tally_streams[i]); cudaStreamWaitEvent(main_stream, ctx->ev_tally[i], 0); }
  };
  for (int k = 0; k < fo->h.num_trees && st == DPHY_OK; ++k) {
    for (int attempt = 0; attempt < 2; ++attempt) {
      st = DPHY_OK;
      if (forked) ctx->stream = ctx->tally_streams[k % kS];        // the per-tree launchers enqueue on ctx->stream
      if (out_Ttwiddle_l) st = tally_times(ctx, fo, k, nullptr, out_Ttwiddle_l + (size_t)k * ld, nullptr, true);
      if (st == DPHY_OK && out_num_muts_l) st = tally_num_muts(ctx, fo, k, nullptr, out_num_muts_l + (size_t)k * ld, nullptr, true);
      ctx->stream = main_stream;
      if (st != DPHY_ERR_OUT_OF_MEMORY || attempt == 1) break;
      // arena full: drain what is in flight, reopen the scope, retry this tree once
      join();
      st = drain();
      if (st != DPHY_OK) break;
      if (forked) { cudaEventRecord(ctx->ev_fork, main_stream); for (int i = 0; i < kS; ++i) cudaStreamWaitEvent(ctx->tally_streams[i], ctx->ev_fork, 0); }
    }
  }
  join();
  const int st2 = drain();
  return st != DPHY_OK ? st : st2;
}

int dphy_forest_calc_Ttwiddle_l(dphy_ctx* ctx, dphy_forest* fo, int32_t tree, double* out_l, double* out_l_a) {
  if (!ctx || !fo || (!out_l && !out_l_a) || tree < 0 || tree >= fo->h.num_trees) return DPHY_ERR_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  return tally_times(ctx, fo, tree, nullptr, out_l, out_l_a);
}

}  // extern "C"
