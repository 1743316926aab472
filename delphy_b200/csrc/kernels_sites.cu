// kernels_sites.cu -- per-site derived tables of a (reference sequence, Global_evo_model) pair (sm_100a).
//
// Replaces calc_cum_Q_l_for_sequence (core/phylo_tree_calc.cpp:379-388) and
// calc_state_frequencies_per_partition_of (core/phylo_tree_calc.cpp:95-106), which the reference recomputes once per
// cycle per Subrun after set_evo (core/subrun.cpp:17-26) and which together were ~18 % of a 200-tip run
// (plans/2026-03-17-01-cache-ref-seq-derived-quantities.md:46-57).  Also builds the tables the tally kernels use:
// munu[l] = mu_{beta(l)} nu_l and the per-(partition, state) cumulative nu tables that turn the reference's
// per-missing-site loops (core/phylo_tree_calc.cpp:309-314) into two table look-ups per interval.
#include "dphy_internal.h"
#include "device_utils.cuh"

#include <cooperative_groups.h>

namespace dphy {

constexpr int kScanThreads = 1024;

// A thread-block cluster of kClusterCtas CTAs sweeps the sites in rounds: CTA r of the cluster takes slab round * kClusterCtas + r
// (kScanThreads * kSitesPerThread consecutive sites; thread tid owns kSitesPerThread consecutive sites, so every load of a warp is
// one contiguous run, summed left to right), scans it, and publishes the slab total into the shared memory of EVERY CTA of the
// cluster (distributed shared memory); after one cluster barrier each CTA adds the totals of the lower ranks and the running
// carry.  L = 29,903 is one round of 8 slabs.  (The reference's scan is strictly sequential; see DESIGN.md section 2.3 for why the
// comparison uses 1e-10.)
namespace cg = cooperative_groups;
constexpr int kSitesPerThread = 4;
constexpr int kClusterCtas = 8;
struct EvoArgs { double mu[kMaxPartitions]; double q[kMaxPartitions * 16]; };   // passed by value: no staging copies

__device__ __forceinline__ void sites_derive_body(
    int L, int P, const uint8_t* __restrict__ ref, const uint8_t* __restrict__ part, const double* __restrict__ nu,
    const EvoArgs& evo, double* __restrict__ munu, double2* __restrict__ munu2, double* __restrict__ cumQ,
    int32_t* __restrict__ ref_freq, double* __restrict__ cum_nu_ba) {
  __shared__ double s_q[kMaxPartitions * 16];
  __shared__ double s_mu[kMaxPartitions];
  __shared__ double s_ws[kScanThreads / 32];
  __shared__ int s_freq[kMaxPartitions * 4];
  __shared__ double s_tot[2][kClusterCtas];      // slab totals of the current exchange, written by every CTA of the cluster
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int tid = threadIdx.x;
  const int K = P * 4;
  if (tid < P * 16) s_q[tid] = evo.q[tid];
  if (tid < P) s_mu[tid] = evo.mu[tid];
  if (tid < kMaxPartitions * 4) s_freq[tid] = 0;
  if (rank == 0 && tid == 0) cumQ[0] = 0.0;
  if (rank == 0 && cum_nu_ba != nullptr && tid < K) cum_nu_ba[(size_t)tid * (L + 1)] = 0.0;
  __syncthreads();
  int cnt[kMaxPartitions * 4];
#pragma unroll
  for (int i = 0; i < kMaxPartitions * 4; ++i) cnt[i] = 0;
  constexpr int kSlab = kScanThreads * kSitesPerThread;
  const int num_slabs = (L + kSlab - 1) / kSlab;
  const int rounds = (num_slabs + kClusterCtas - 1) / kClusterCtas;
  int xchg = 0;                                  // exchanges so far (parity selects the s_tot buffer)
  double carry = 0.0;                            // sum of every slab of the earlier rounds (identical in all CTAs)
  double carry_k[kMaxPartitions * 4];
#pragma unroll
  for (int i = 0; i < kMaxPartitions * 4; ++i) carry_k[i] = 0.0;

  // one exchange: block scan of `t`, totals to every CTA, cluster barrier; returns the exclusive prefix of this thread's first
  // site within the round (lower ranks + own lower threads) and the round's grand total
  auto exchange = [&](double t, double& round_total) -> double {
    double bt;
    __syncthreads();                             // s_ws may still be read from the previous scan
    const double incl = block_scan_incl<double, kScanThreads>(t, s_ws, &bt);
    const int par = xchg & 1; ++xchg;
    if (tid < kClusterCtas) *cluster.map_shared_rank(&s_tot[par][rank], tid) = bt;     // my total into CTA tid's buffer
    cluster.sync();
    double lower = 0.0, all = 0.0;
#pragma unroll
    for (int r = 0; r < kClusterCtas; ++r) { const double x = s_tot[par][r]; if (r < rank) lower += x; all += x; }
    round_total = all;
    return lower + (incl - t);
  };

  for (int round = 0; round < rounds; ++round) {
    const int l0 = (round * kClusterCtas + rank) * kSlab + tid * kSitesPerThread;
    double v[kSitesPerThread], nuv[kSitesPerThread];
    int key[kSitesPerThread];
    double tot = 0.0;
#pragma unroll
    for (int u = 0; u < kSitesPerThread; ++u) {
      const int l = l0 + u;
      v[u] = 0.0; nuv[u] = 0.0; key[u] = -1;
      if (l < L) {
        const int pt = part[l], a = ref[l];
        nuv[u] = nu[l]; key[u] = pt * 4 + a;
        const double mn = s_mu[pt] * nuv[u];
        munu[l] = mn;
        if (munu2 != nullptr) munu2[l] = make_double2(mn, log(mn));      // site-rate heterogeneity: the log of every mutation's rate, once per site
        v[u] = mn * (-s_q[pt * 16 + a * 5]);
#pragma unroll
        for (int i = 0; i < kMaxPartitions * 4; ++i) cnt[i] += (i == key[u]);
      }
      tot += v[u];
    }
    double all;
    double run = carry + exchange(tot, all);     // exclusive prefix of my first site
    carry += all;
#pragma unroll
    for (int u = 0; u < kSitesPerThread; ++u) {
      run += v[u];
      if (l0 + u < L) cumQ[l0 + u + 1] = run;
    }
    // cumulative nu per (partition, state): cum_nu_ba[(b*4+a)*(L+1) + l] = sum_{l' < l, beta(l')=b, ref[l']=a} nu_l'  (same sweep;
    // depends on nu_l alone, so it is skipped when only mu / pi / q changed)
    if (cum_nu_ba != nullptr) {
#pragma unroll
      for (int k = 0; k < kMaxPartitions * 4; ++k) {
        if (k < K) {
          double t = 0.0;
#pragma unroll
          for (int u = 0; u < kSitesPerThread; ++u) t += key[u] == k ? nuv[u] : 0.0;
          double allk;
          double r = carry_k[k] + exchange(t, allk);
          carry_k[k] += allk;
          double* out = cum_nu_ba + (size_t)k * (L + 1);
#pragma unroll
          for (int u = 0; u < kSitesPerThread; ++u) {
            if (key[u] == k) r += nuv[u];
            if (l0 + u < L) out[l0 + u + 1] = r;
          }
        }
      }
    }
  }
  // reference-state counts: every CTA adds its own into rank 0's shared memory
#pragma unroll
  for (int i = 0; i < kMaxPartitions * 4; ++i) if (cnt[i]) atomicAdd(cluster.map_shared_rank(&s_freq[i], 0), cnt[i]);
  cluster.sync();
  if (rank == 0 && tid < P * 4) ref_freq[tid] = s_freq[tid];
}

__global__ void __cluster_dims__(kClusterCtas, 1, 1) __launch_bounds__(kScanThreads) sites_derive_kernel(
    int L, int P, const uint8_t* __restrict__ ref, const uint8_t* __restrict__ part, const double* __restrict__ nu,
    const __grid_constant__ EvoArgs evo, double* __restrict__ munu, double2* __restrict__ munu2, double* __restrict__ cumQ,
    int32_t* __restrict__ ref_freq, double* __restrict__ cum_nu_ba) {
  sites_derive_body(L, P, ref, part, nu, evo, munu, munu2, cumQ, ref_freq, cum_nu_ba);
}

// The same for MANY tables in one launch: cluster c derives table c.  What Run::push_global_params_to_subruns does once per cycle
// (core/run.cpp:267-275: the new mu / pi / q go to every subrun's evo model): sixteen 13-us launches of one cluster each leave
// 140 of the 148 SMs idle sixteen times over.
struct DeriveArgs {
  int32_t L, P;
  const uint8_t* ref; const uint8_t* part; const double* nu;
  double* munu; double2* munu2; double* cumQ; int32_t* ref_freq; double* cum_nu_ba;
  EvoArgs evo;
};
__global__ void __cluster_dims__(kClusterCtas, 1, 1) __launch_bounds__(kScanThreads) sites_derive_many_kernel(const DeriveArgs* __restrict__ args) {
  const DeriveArgs& a = args[blockIdx.x / kClusterCtas];
  sites_derive_body(a.L, a.P, a.ref, a.part, a.nu, a.evo, a.munu, a.munu2, a.cumQ, a.ref_freq, a.cum_nu_ba);
}

// Cumulative reference-state counts per (partition, state), interleaved by site:
// cref[l*(4P) + b*4+a] = #{l' < l : beta(l') == b, ref[l'] == a}  (one 16-byte look-up per partition and interval end).
// Structure only (reference sequence + partition map), so it is built once per sites table.  One CTA per (b, a) row.
// fold_branch_weights_kernel uses it to turn a missation interval into the 4P state counts of the sites it hides.
__global__ void __launch_bounds__(kScanThreads) sites_ref_counts_kernel(int L, const uint8_t* __restrict__ ref,
                                                                        const uint8_t* __restrict__ part, int32_t* __restrict__ cref) {
  __shared__ int s_ws[kScanThreads / 32];
  const int k = blockIdx.x, tid = threadIdx.x;
  const int chunk = (L + kScanThreads - 1) / kScanThreads;
  const int l0 = min(tid * chunk, L), l1 = min(l0 + chunk, L);
  int c = 0;
  for (int l = l0; l < l1; ++l) c += (part[l] * 4 + ref[l] == k);
  int tot;
  const int incl = block_scan_incl<int, kScanThreads>(c, s_ws, &tot);
  int run = incl - c;
  const size_t K = gridDim.x;
  if (tid == 0) cref[k] = 0;
  for (int l = l0; l < l1; ++l) {
    run += (part[l] * 4 + ref[l] == k);
    cref[(size_t)(l + 1) * K + k] = run;
  }
}

int launch_sites_ref_counts(dphy_ctx* ctx, dphy_sites* s) {
  sites_ref_counts_kernel<<<s->P * 4, kScanThreads, 0, ctx->stream>>>(s->L, s->d_ref, s->d_part, s->d_cref);
  ctx->launches += 1;
  return check_cuda(ctx, cudaGetLastError(), "sites_ref_counts_kernel launch");
}

// with_nu_tables: also rebuild the cumulative-nu tables (they depend on nu_l alone: skipped when only mu / pi / q changed)
int launch_sites_derive(dphy_ctx* ctx, dphy_sites* s, bool with_nu_tables) {
  EvoArgs evo;
  for (int i = 0; i < kMaxPartitions; ++i) evo.mu[i] = s->h.mu[i];
  for (int i = 0; i < kMaxPartitions * 16; ++i) evo.q[i] = s->h.q[i];
  sites_derive_kernel<<<kClusterCtas, kScanThreads, 0, ctx->stream>>>(s->L, s->P, s->d_ref, s->d_part, s->d_nu, evo, s->d_munu,
                                                           s->h.nu_uniform ? nullptr : s->d_munu2, s->d_cumQ, s->d_ref_freq, with_nu_tables ? s->d_cum_nu_ba : nullptr);
  ctx->launches += 1;
  return check_cuda(ctx, cudaGetLastError(), "sites_derive_kernel launch");
}

// mu / pi / q changed on every table of `tables` (site rates untouched): one launch, one cluster per table
int launch_sites_derive_many(dphy_ctx* ctx, dphy_sites* const* tables, int n) {
  if (n <= 0) return DPHY_OK;
  PinnedStage pin(ctx, sizeof(DeriveArgs) * (size_t)n);
  if (pin.status != DPHY_OK) return pin.status;
  DeriveArgs* h = reinterpret_cast<DeriveArgs*>(pin.p);
  for (int k = 0; k < n; ++k) {
    dphy_sites* s = tables[k];
    DeriveArgs& a = h[k];
    a.L = s->L; a.P = s->P; a.ref = s->d_ref; a.part = s->d_part; a.nu = s->d_nu;
    a.munu = s->d_munu; a.munu2 = s->h.nu_uniform ? nullptr : s->d_munu2; a.cumQ = s->d_cumQ; a.ref_freq = s->d_ref_freq; a.cum_nu_ba = nullptr;
    for (int i = 0; i < kMaxPartitions; ++i) a.evo.mu[i] = s->h.mu[i];
    for (int i = 0; i < kMaxPartitions * 16; ++i) a.evo.q[i] = s->h.q[i];
  }
  const size_t mark = ctx->arena.mark();
  DeriveArgs* d = static_cast<DeriveArgs*>(ctx->arena.alloc(sizeof(DeriveArgs) * (size_t)n));
  if (!d) { ctx->arena.release(mark); return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "arena exhausted (set_evo_many)"); }
  cudaError_t ce = cudaMemcpyAsync(d, h, sizeof(DeriveArgs) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream);
  pin.reset();
  if (ce == cudaSuccess) {
    sites_derive_many_kernel<<<kClusterCtas * n, kScanThreads, 0, ctx->stream>>>(d);
    ctx->launches += 1;
    ce = cudaGetLastError();
  }
  ctx->arena.release(mark);      // (the next user of the arena enqueues behind this launch on the same stream)
  return check_cuda(ctx, ce, "sites_derive_many_kernel launch");
}

}  // namespace dphy
