// c_abi.cu -- host side of the C ABI declared in include/delphy_b200.h: context, device arena, upload of the
// flattened EMATs (host node order -> device DFS order), result download.  No CPU fallback anywhere: if CUDA is not
// usable every compute entry point fails with DPHY_ERR_CUDA.
#include "dphy_internal.h"

#include <algorithm>
#include <atomic>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include <thread>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <limits>
#include <memory>
#include <new>

namespace dphy {

int set_error(dphy_ctx* ctx, int status, const std::string& msg) {
  if (ctx) ctx->last_error = msg;
  return status;
}
int check_cuda(dphy_ctx* ctx, cudaError_t e, const char* what) {
  if (e == cudaSuccess) return DPHY_OK;
  return set_error(ctx, DPHY_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

// Pinned staging buffer owned by the ctx, grown geometrically.  Copies out of it are asynchronous: the next user waits
// on the event recorded by release_pinned_async() instead of synchronizing the whole stream.
int acquire_pinned(dphy_ctx* ctx, size_t bytes, void** out) {
  if (ctx->pinned_in_flight) { cudaEventSynchronize(ctx->pinned_ev); ctx->pinned_in_flight = false; }
  if (ctx->pinned_bytes < bytes) {
    if (ctx->pinned) { cudaFreeHost(ctx->pinned); ctx->pinned = nullptr; ctx->pinned_bytes = 0; }
    size_t want = std::max(bytes, (size_t)1 << 20);
    DPHY_CUDA(ctx, cudaMallocHost(&ctx->pinned, want));
    ctx->pinned_bytes = want;
  }
  *out = ctx->pinned;
  return DPHY_OK;
}
void release_pinned_async(dphy_ctx* ctx) {
  if (cudaEventRecord(ctx->pinned_ev, ctx->stream) == cudaSuccess) ctx->pinned_in_flight = true;
  else cudaStreamSynchronize(ctx->stream);
}

// Forests hold a device copy of each SitesDev record; re-sync it after dphy_sites_set_evo changed mu/pi/q.
int refresh_sites(dphy_ctx* ctx, dphy_forest* fo) {
  for (size_t i = 0; i < fo->sites.size(); ++i) {
    if (fo->sites_version[i] != fo->sites[i]->version) {
      DPHY_CUDA(ctx, cudaMemcpyAsync(const_cast<SitesDev*>(fo->h.sites) + i, &fo->sites[i]->h, sizeof(SitesDev),
                                     cudaMemcpyHostToDevice, ctx->stream));
      fo->sites_version[i] = fo->sites[i]->version;
    }
  }
  return DPHY_OK;
}
}  // namespace dphy

using namespace dphy;

extern "C" {

const char* dphy_version(void) { return "delphy_b200 0.1 (sm_100a)"; }

int dphy_host_alloc(dphy_ctx* ctx, size_t bytes, void** out) {
  if (!ctx || !out) return DPHY_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  cudaSetDevice(ctx->device);
  if (cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError();
    return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaHostAlloc");
  }
  return DPHY_OK;
}
void dphy_host_free(dphy_ctx* ctx, void* p) {
  if (ctx) cudaSetDevice(ctx->device);
  if (p) cudaFreeHost(p);
}

int dphy_ctx_create(int device, dphy_ctx** out) {
  if (!out) return DPHY_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0 || device < 0 || device >= count) {
    return DPHY_ERR_CUDA;   // no CPU fallback: the product path requires a CUDA device
  }
  auto* ctx = new (std::nothrow) dphy_ctx();
  if (!ctx) return DPHY_ERR_OUT_OF_MEMORY;
  ctx->device = device;
  if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return DPHY_ERR_CUDA; }
  // the main stream outranks the library's side streams (created at the default, lowest priority): where a bandwidth-bound tail
  // kernel of one SPR batch runs next to the latency-bound set-up chain of the next, freed SM slots go to the chain first
  {
    int prio_least = 0, prio_greatest = 0;
    cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
    if (cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_greatest) != cudaSuccess) { delete ctx; return DPHY_ERR_CUDA; }
  }
  if (cudaEventCreateWithFlags(&ctx->pinned_ev, cudaEventDisableTiming) != cudaSuccess) { cudaStreamDestroy(ctx->stream); delete ctx; return DPHY_ERR_CUDA; }
  // keep freed stream-ordered allocations cached in the pool (no cudaMalloc on the hot path after warm-up)
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    uint64_t thr = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  ctx->arena.capacity = (size_t)256 << 20;
  if (cudaMalloc((void**)&ctx->arena.base, ctx->arena.capacity) != cudaSuccess) {
    cudaStreamDestroy(ctx->stream); delete ctx; return DPHY_ERR_OUT_OF_MEMORY;
  }
  *out = ctx;
  return DPHY_OK;
}

void dphy_ctx_destroy(dphy_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->arena.base) cudaFree(ctx->arena.base);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  if (ctx->aux_stream) { cudaStreamSynchronize(ctx->aux_stream); cudaStreamDestroy(ctx->aux_stream); }
  if (ctx->tail_stream) { cudaStreamSynchronize(ctx->tail_stream); cudaStreamDestroy(ctx->tail_stream); }
  for (auto& blk : ctx->spr_blocks) { if (blk.ev) cudaEventDestroy(blk.ev); cudaFree(blk.ptr); }
  if (ctx->ev_tail) cudaEventDestroy(ctx->ev_tail);
  for (int i = 0; i < dphy_ctx::kTallyStreams; ++i) {
    if (ctx->tally_streams[i]) { cudaStreamSynchronize(ctx->tally_streams[i]); cudaStreamDestroy(ctx->tally_streams[i]); }
    if (ctx->ev_tally[i]) cudaEventDestroy(ctx->ev_tally[i]);
  }
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  if (ctx->pinned_ev) cudaEventDestroy(ctx->pinned_ev);
  if (ctx->copy_stream) {
    cudaStreamSynchronize(ctx->copy_stream);
    cudaEventDestroy(ctx->ev_main); cudaEventDestroy(ctx->ev_topo); cudaEventDestroy(ctx->ev_nodes); cudaEventDestroy(ctx->ev_lists);
    for (cudaEvent_t e : ctx->ev_tree) cudaEventDestroy(e);
    for (int i = 0; i < dphy_ctx::kCopyStreams; ++i) {
      if (ctx->copy_streams[i]) { cudaStreamSynchronize(ctx->copy_streams[i]); cudaStreamDestroy(ctx->copy_streams[i]); }
      if (ctx->ev_copy[i]) cudaEventDestroy(ctx->ev_copy[i]);
    }
  }
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* dphy_last_error(const dphy_ctx* ctx) { return ctx ? ctx->last_error.c_str() : "no context (CUDA device unavailable?)"; }

int dphy_ctx_join_side_streams(dphy_ctx* ctx) {
  if (!ctx) return DPHY_ERR_INVALID_ARGUMENT;
  if (ctx->tail_stream && ctx->tail_dirty) {
    cudaSetDevice(ctx->device);
    DPHY_CUDA(ctx, cudaEventRecord(ctx->ev_tail, ctx->tail_stream));
    DPHY_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_tail, 0));
    ctx->tail_dirty = false;
  }
  return DPHY_OK;
}

int dphy_ctx_synchronize(dphy_ctx* ctx) {
  if (!ctx) return DPHY_ERR_INVALID_ARGUMENT;
  int st = dphy_ctx_join_side_streams(ctx);
  if (st != DPHY_OK) return st;
  DPHY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return DPHY_OK;
}

int dphy_arena_stats(const dphy_ctx* ctx, size_t* capacity, size_t* high_water) {
  if (!ctx) return DPHY_ERR_INVALID_ARGUMENT;
  if (capacity) *capacity = ctx->arena.capacity;
  if (high_water) *high_water = ctx->arena.high_water;
  return DPHY_OK;
}

int dphy_ctx_set_log_G_path(dphy_ctx* ctx, int path) {
  if (!ctx || (path != DPHY_LOG_G_PATH_AUTO && path != DPHY_LOG_G_PATH_GENERAL)) return DPHY_ERR_INVALID_ARGUMENT;
  ctx->logg_path = path;
  return DPHY_OK;
}

void* dphy_ctx_stream(dphy_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
int64_t dphy_ctx_launch_count(const dphy_ctx* ctx) { return ctx ? ctx->launches : 0; }

// ---- sites ------------------------------------------------------------------------------------------------------
static void set_nu_uniform(dphy_sites* s, const double* nu_l) {
  // no site-rate heterogeneity <=> every nu_l equals the same constant: mu*nu needs no per-site gather
  bool uni = true;
  for (int l = 1; l < s->L && uni; ++l) uni = (nu_l[l] == nu_l[0]);
  s->h.nu_uniform = uni ? 1 : 0;
  s->h.nu_const = uni ? nu_l[0] : 1.0;
  s->h.pad = 0;
}

static void fill_tables(dphy_sites* s) {
  for (int i = 0; i < kMaxPartitions * 16; ++i) {
    const int pt = i >> 4, x = (i >> 2) & 3, y = i & 3;
    if (pt < s->P) {
      const double dq = (-s->h.q[pt * 16 + y * 5]) - (-s->h.q[pt * 16 + x * 5]);
      s->h.tab_dq[i] = dq;
      s->h.tab_md[i] = s->h.mu[pt] * s->h.nu_const * dq;
      s->h.tab_lq[i] = x != y ? std::log(s->h.mu[pt] * s->h.nu_const * s->h.q[i]) : 0.0;
      s->h.tab_logq[i] = x != y ? std::log(s->h.q[i]) : 0.0;
    } else {
      s->h.tab_dq[i] = 0.0; s->h.tab_md[i] = 0.0; s->h.tab_lq[i] = 0.0; s->h.tab_logq[i] = 0.0;
    }
  }
  for (int i = 0; i < kMaxPartitions * 4; ++i) {
    const int pt = i >> 2, a = i & 3;
    s->h.tab_muq[i] = pt < s->P ? s->h.mu[pt] * s->h.nu_const * (-s->h.q[pt * 16 + a * 5]) : 0.0;
  }
}

// Validate first, commit second: a rejected model must leave the host mirror untouched (no half-updated tables).
static int validate_evo(dphy_ctx* ctx, int P, int L, const double* nu_l, const double* mu, const double* pi_a, const double* q_ab) {
  for (int b = 0; b < P; ++b) {
    if (!(mu[b] >= 0.0) || !std::isfinite(mu[b])) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "mu must be finite and >= 0");
    for (int a = 0; a < 4; ++a) {
      if (!(pi_a[b * 4 + a] >= 0.0) || !std::isfinite(pi_a[b * 4 + a])) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "pi_a must be finite and >= 0");
      for (int c = 0; c < 4; ++c) {
        const double q = q_ab[b * 16 + a * 4 + c];
        if (!std::isfinite(q) || (a != c && q < 0.0) || (a == c && q > 0.0)) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "q_ab must be a finite rate matrix (off-diagonal >= 0, diagonal <= 0)");
      }
    }
  }
  if (nu_l) for (int l = 0; l < L; ++l) if (!(nu_l[l] >= 0.0) || !std::isfinite(nu_l[l])) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "nu_l must be finite and >= 0");
  return DPHY_OK;
}

static void fill_evo(dphy_sites* s, const double* mu, const double* pi_a, const double* q_ab) {
  for (int b = 0; b < s->P; ++b) {
    s->h.mu[b] = mu[b];
    for (int a = 0; a < 4; ++a) {
      s->h.pi[b * 4 + a] = pi_a[b * 4 + a];
      for (int c = 0; c < 4; ++c) s->h.q[b * 16 + a * 4 + c] = q_ab[b * 16 + a * 4 + c];
    }
  }
}

static int validate_sequence(dphy_ctx* ctx, const dphy_sites_host* host) {
  const int L = host->num_sites, P = host->num_partitions;
  for (int l = 0; l < L; ++l) {
    if (host->ref[l] > 3) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "ref_sequence holds a non-ACGT state");
    if (host->partition_for_site[l] < 0 || host->partition_for_site[l] >= P)
      return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "partition_for_site out of range");
  }
  return DPHY_OK;
}

// stage ref / partition / nu through the pinned slab and re-derive every table (stream-ordered)
static int upload_sequence_and_derive(dphy_ctx* ctx, dphy_sites* s, const dphy_sites_host* host) {
  const int L = s->L;
  const size_t off_part = align_up(L), off_nu = 2 * off_part, total = off_nu + sizeof(double) * (size_t)L;
  PinnedStage pin(ctx, total);
  if (pin.status != DPHY_OK) return pin.status;
  char* hb = pin.p;
  std::memcpy(hb, host->ref, L);
  uint8_t* hp = reinterpret_cast<uint8_t*>(hb + off_part);
  for (int l = 0; l < L; ++l) hp[l] = (uint8_t)host->partition_for_site[l];
  std::memcpy(hb + off_nu, host->nu_l, sizeof(double) * L);
  set_nu_uniform(s, host->nu_l);
  fill_tables(s);
  cudaError_t e = cudaMemcpyAsync(s->d_ref, hb, L, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(s->d_part, hb + off_part, L, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(s->d_nu, hb + off_nu, sizeof(double) * L, cudaMemcpyHostToDevice, ctx->stream);
  pin.reset();
  if (e != cudaSuccess) return check_cuda(ctx, e, "H2D sites");
  int st = launch_sites_derive(ctx, s);
  if (st == DPHY_OK) st = launch_sites_ref_counts(ctx, s);
  return st;
}

int dphy_sites_upload(dphy_ctx* ctx, const dphy_sites_host* host, dphy_sites** out) {
  if (!ctx || !host || !out) return DPHY_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  const int L = host->num_sites, P = host->num_partitions;
  if (L <= 0) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "num_sites must be > 0");
  if (P <= 0 || P > kMaxPartitions) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "num_partitions must be in [1,4]");
  int st = validate_sequence(ctx, host);
  if (st == DPHY_OK) st = validate_evo(ctx, P, L, host->nu_l, host->mu, host->pi_a, host->q_ab);
  if (st != DPHY_OK) return st;
  std::unique_ptr<dphy_sites> s(new (std::nothrow) dphy_sites());
  if (!s) return DPHY_ERR_OUT_OF_MEMORY;
  s->L = L; s->P = P;
  fill_evo(s.get(), host->mu, host->pi_a, host->q_ab);
  cudaSetDevice(ctx->device);
  Slab slab;
  const int b_ref = slab.reserve(L), b_part = slab.reserve(L), b_nu = slab.reserve(sizeof(double) * L);
  const int b_munu = slab.reserve(sizeof(double) * L), b_cumQ = slab.reserve(sizeof(double) * (L + 1));
  const int b_munu2 = slab.reserve(sizeof(double2) * L);
  const int b_freq = slab.reserve(sizeof(int32_t) * kMaxPartitions * 4);
  const int b_cnu = slab.reserve(sizeof(double) * (size_t)P * 4 * (L + 1));
  const int b_cref = slab.reserve(sizeof(int32_t) * (size_t)P * 4 * (L + 1));
  // stream-ordered pool allocation: no device-wide synchronization, and a freed table's block is reused by the next one
  DevBlock blk(ctx->stream);
  if (!blk.alloc(slab.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(sites)");
  char* dbase = blk.p;
  s->bytes = slab.total;
  s->d_ref = slab.at<uint8_t>(dbase, b_ref); s->d_part = slab.at<uint8_t>(dbase, b_part); s->d_nu = slab.at<double>(dbase, b_nu);
  s->d_munu = slab.at<double>(dbase, b_munu); s->d_cumQ = slab.at<double>(dbase, b_cumQ);
  s->d_munu2 = slab.at<double2>(dbase, b_munu2); s->h.munu2 = s->d_munu2;
  s->d_ref_freq = slab.at<int32_t>(dbase, b_freq); s->d_cum_nu_ba = slab.at<double>(dbase, b_cnu);
  s->d_cref = slab.at<int32_t>(dbase, b_cref);
  s->h.L = L; s->h.P = P; s->h.ref = s->d_ref; s->h.part = s->d_part; s->h.nu = s->d_nu; s->h.munu = s->d_munu;
  s->h.cumQ = s->d_cumQ; s->h.ref_freq = s->d_ref_freq; s->h.cref = s->d_cref;
  st = upload_sequence_and_derive(ctx, s.get(), host);
  if (st != DPHY_OK) return st;
  blk.release();                // s->d_ref is the block's base
  *out = s.release();
  return DPHY_OK;
}

int dphy_sites_update(dphy_ctx* ctx, dphy_sites* s, const dphy_sites_host* host) {
  if (ctx) dphy_ctx_join_side_streams(ctx);
  if (!ctx || !s || !host) return DPHY_ERR_INVALID_ARGUMENT;
  if (host->num_sites != s->L || host->num_partitions != s->P) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "sites update: number of sites / partitions differs from the table's");
  int st = validate_sequence(ctx, host);
  if (st == DPHY_OK) st = validate_evo(ctx, s->P, s->L, host->nu_l, host->mu, host->pi_a, host->q_ab);
  if (st != DPHY_OK) return st;
  cudaSetDevice(ctx->device);
  fill_evo(s, host->mu, host->pi_a, host->q_ab);
  s->version += 1;
  return upload_sequence_and_derive(ctx, s, host);
}

void dphy_sites_destroy(dphy_ctx* ctx, dphy_sites* s) {
  if (ctx) dphy_ctx_join_side_streams(ctx);
  if (!s) return;
  if (s->d_ref) {   // base of the slab
    if (ctx) { cudaSetDevice(ctx->device); cudaFreeAsync(s->d_ref, ctx->stream); }   // stream-ordered: after the last kernel that reads it
    else cudaFree(s->d_ref);
  }
  delete s;
}

int dphy_sites_set_evo(dphy_ctx* ctx, dphy_sites* s, const double* nu_l, const double* mu, const double* pi_a, const double* q_ab) {
  if (!ctx || !s || !mu || !pi_a || !q_ab) return DPHY_ERR_INVALID_ARGUMENT;
  int st = validate_evo(ctx, s->P, s->L, nu_l, mu, pi_a, q_ab);
  if (st != DPHY_OK) return st;
  fill_evo(s, mu, pi_a, q_ab);
  if (nu_l) {
    PinnedStage pin(ctx, sizeof(double) * s->L);
    if (pin.status != DPHY_OK) return pin.status;
    std::memcpy(pin.p, nu_l, sizeof(double) * s->L);
    set_nu_uniform(s, nu_l);
    DPHY_CUDA(ctx, cudaMemcpyAsync(s->d_nu, pin.p, sizeof(double) * s->L, cudaMemcpyHostToDevice, ctx->stream));
  }
  fill_tables(s);
  s->version += 1;
  // asynchronous: everything that consumes the tables is ordered after this on the ctx's stream, and the forests pick up the
  // new host-side constants (mu, q, the 64-entry event tables) through the version bump
  return launch_sites_derive(ctx, s, /*with_nu_tables=*/nu_l != nullptr);
}

int dphy_sites_set_evo_many(dphy_ctx* ctx, int32_t n, dphy_sites* const* tables, const double* const* mu, const double* const* pi_a,
                            const double* const* q_ab) {
  if (!ctx || n < 0 || (n > 0 && (!tables || !mu || !pi_a || !q_ab))) return DPHY_ERR_INVALID_ARGUMENT;
  // validate everything before anything is committed
  for (int k = 0; k < n; ++k) {
    if (!tables[k] || !mu[k] || !pi_a[k] || !q_ab[k]) return DPHY_ERR_INVALID_ARGUMENT;
    for (int j = 0; j < k; ++j) if (tables[j] == tables[k]) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "set_evo_many: a table is listed twice");
    const int st = validate_evo(ctx, tables[k]->P, tables[k]->L, nullptr, mu[k], pi_a[k], q_ab[k]);
    if (st != DPHY_OK) return st;
  }
  cudaSetDevice(ctx->device);
  for (int k = 0; k < n; ++k) {
    fill_evo(tables[k], mu[k], pi_a[k], q_ab[k]);
    fill_tables(tables[k]);
    tables[k]->version += 1;
  }
  return launch_sites_derive_many(ctx, tables, n);
}

int dphy_calc_state_frequencies_per_partition(dphy_ctx* ctx, dphy_sites* s, int32_t* out) {
  if (!ctx || !s || !out) return DPHY_ERR_INVALID_ARGUMENT;
  DPHY_CUDA(ctx, cudaMemcpyAsync(out, s->d_ref_freq, sizeof(int32_t) * s->P * 4, cudaMemcpyDeviceToHost, ctx->stream));
  return check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "state frequencies D2H");
}

int dphy_calc_cum_Q_l(dphy_ctx* ctx, dphy_sites* s, double* out) {
  if (!ctx || !s || !out) return DPHY_ERR_INVALID_ARGUMENT;
  DPHY_CUDA(ctx, cudaMemcpyAsync(out, s->d_cumQ, sizeof(double) * (s->L + 1), cudaMemcpyDeviceToHost, ctx->stream));
  return check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "cum_Q_l D2H");
}

// ---- forest -------------------------------------------------------------------------------------------------------
namespace {

// Host -> device copy of many caller-owned (pageable) arrays: worker threads memcpy 2 MiB chunks into the pinned
// staging slab while the main thread issues the H2D DMA of every finished chunk, so the memcpy and the PCIe transfer
// overlap and the host never touches the data more than once.
struct CopyJob { size_t dst_off; const void* src; size_t bytes; int group; int tree; };   // group 0: topology (needed first), 1: node times + offsets, 2: lists

// Host copy into the pinned staging slab with non-temporal stores: the destination is read next by the DMA engine, not by this
// core, so it should neither be fetched for ownership nor displace the source from the cache (plain memcpy below 16 bytes or
// on non-SSE2 hosts).
void stream_copy(char* dst, const char* src, size_t n) {
#if defined(__SSE2__)
  if (n >= 256) {
    const size_t head = (16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15;
    if (head) { std::memcpy(dst, src, head); dst += head; src += head; n -= head; }
    const size_t blocks = n / 64;
    for (size_t i = 0; i < blocks; ++i) {
      const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src) + 0), b = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src) + 1);
      const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src) + 2), d = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src) + 3);
      _mm_stream_si128(reinterpret_cast<__m128i*>(dst) + 0, a); _mm_stream_si128(reinterpret_cast<__m128i*>(dst) + 1, b);
      _mm_stream_si128(reinterpret_cast<__m128i*>(dst) + 2, c); _mm_stream_si128(reinterpret_cast<__m128i*>(dst) + 3, d);
      src += 64; dst += 64;
    }
    n -= blocks * 64;
    _mm_sfence();
  }
#endif
  if (n) std::memcpy(dst, src, n);
}

// page-locked host memory or device memory: the copy engine can read it where it lies
bool is_pinned_host(const void* p) {
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeDevice;
}

void sync_copy_streams(dphy_ctx* ctx) {
  for (int i = 0; i < dphy_ctx::kCopyStreams; ++i) if (ctx->copy_streams[i]) cudaStreamSynchronize(ctx->copy_streams[i]);
}

int ensure_copy_stream(dphy_ctx* ctx) {
  if (ctx->copy_stream) return DPHY_OK;
  for (int i = 0; i < dphy_ctx::kCopyStreams; ++i) {
    DPHY_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->copy_streams[i], cudaStreamNonBlocking));
    DPHY_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_copy[i], cudaEventDisableTiming));
  }
  ctx->copy_stream = ctx->copy_streams[0];
  DPHY_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_main, cudaEventDisableTiming));
  DPHY_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_topo, cudaEventDisableTiming));
  DPHY_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_nodes, cudaEventDisableTiming));
  DPHY_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_lists, cudaEventDisableTiming));
  return DPHY_OK;
}

// *two_phase is set when the copies went to ctx->copy_stream: ev_topo fires once the group-0 arrays (and every byte no job
// covers) have landed, ev_lists once everything has.
int staged_upload(dphy_ctx* ctx, char* pinned, std::vector<CopyJob>& jobs, char* d_base, size_t total, bool* two_phase) {
  *two_phase = false;
  if (total == 0) return DPHY_OK;
  constexpr size_t kChunk = (size_t)2 << 20;
  const size_t nchunks = (total + kChunk - 1) / kChunk;
  std::sort(jobs.begin(), jobs.end(), [](const CopyJob& a, const CopyJob& b) { return a.dst_off < b.dst_off; });
  // Caller arrays that are already page-locked (dphy_host_alloc / cudaHostRegister) are DMA'd from where they lie: no host
  // copy at all.  Only the bytes no job covers (the records written into the staging slab, alignment gaps) come from it.
  {
    bool all_pinned = !jobs.empty();
    for (const CopyJob& j : jobs) if (!is_pinned_host(j.src)) { all_pinned = false; break; }
    if (all_pinned) {
      int st = ensure_copy_stream(ctx);
      if (st != DPHY_OK) return st;
      constexpr int kS = dphy_ctx::kCopyStreams;
      cudaStream_t cs = ctx->copy_stream;
      // the destination was allocated stream-ordered on the main stream: ev_main was recorded right after that allocation (the
      // slab memsets that follow it there touch other memory and need not delay the DMA)
      cudaError_t ce = cudaSuccess;
      for (int i = 0; i < kS; ++i) if (ce == cudaSuccess) ce = cudaStreamWaitEvent(ctx->copy_streams[i], ctx->ev_main, 0);
      int flip = 0;
      auto copy = [&](char* dst, const void* src, size_t bytes) {
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, ctx->copy_streams[flip++ % kS]);
      };
      auto close_group = [&](cudaEvent_t ev) {   // ev fires once every copy stream has drained what was issued so far
        for (int i = 1; i < kS; ++i) {
          if (ce == cudaSuccess) ce = cudaEventRecord(ctx->ev_copy[i], ctx->copy_streams[i]);
          if (ce == cudaSuccess) ce = cudaStreamWaitEvent(cs, ctx->ev_copy[i], 0);
        }
        if (ce == cudaSuccess) ce = cudaEventRecord(ev, cs);
      };
      // (everything meaningful is covered by a job -- the per-tree records written into the staging slab are one -- so the
      // alignment gaps between the destination blocks are not copied)
      for (const CopyJob& j : jobs) if (j.group == 0) copy(d_base + j.dst_off, j.src, j.bytes);   // per-tree records + topology
      close_group(ctx->ev_topo);
      for (const CopyJob& j : jobs) if (j.group == 1) copy(d_base + j.dst_off, j.src, j.bytes);   // node times + CSR offsets
      close_group(ctx->ev_nodes);
      // the bulky per-event arrays, tree by tree (the jobs are sorted by destination, i.e. tree-major): each tree gets its own event
      int cur_tree = -1;
      for (const CopyJob& j : jobs) {
        if (j.group != 2) continue;
        if (j.tree != cur_tree) {
          if (cur_tree >= 0) close_group(ctx->ev_tree[cur_tree]);
          cur_tree = j.tree;
        }
        copy(d_base + j.dst_off, j.src, j.bytes);
      }
      if (cur_tree >= 0) close_group(ctx->ev_tree[cur_tree]);
      close_group(ctx->ev_lists);
      *two_phase = ce == cudaSuccess;
      if (ce != cudaSuccess) for (int i = 0; i < kS; ++i) cudaStreamSynchronize(ctx->copy_streams[i]);   // nothing may still be writing when the caller frees the destination
      return check_cuda(ctx, ce, "H2D direct upload");
    }
  }
  auto fill_chunk = [&](size_t c) {
    const size_t lo = c * kChunk, hi = std::min(total, lo + kChunk);
    // first job that may overlap [lo, hi)
    size_t j = std::upper_bound(jobs.begin(), jobs.end(), lo, [](size_t v, const CopyJob& b) { return v < b.dst_off; }) - jobs.begin();
    if (j > 0) --j;
    for (; j < jobs.size() && jobs[j].dst_off < hi; ++j) {
      const size_t a = std::max(lo, jobs[j].dst_off), b = std::min(hi, jobs[j].dst_off + jobs[j].bytes);
      const char* src = static_cast<const char*>(jobs[j].src) + (a - jobs[j].dst_off);
      if (a < b && src != pinned + a) stream_copy(pinned + a, src, b - a);   // (the per-tree records already lie in the slab)
    }
  };
  unsigned hw = std::thread::hardware_concurrency();
  const size_t nthreads = std::min<size_t>({nchunks, hw ? hw : 1u, (size_t)16});
  // The chunk DMAs go to the copy stream; the same stage events as on the direct path are recorded as soon as the chunk that
  // completes a group (or a tree's lists) has been issued -- the destination layout is group-major for exactly this.
  {
    int st = ensure_copy_stream(ctx);
    if (st != DPHY_OK) return st;
  }
  cudaStream_t cs = ctx->copy_stream;
  struct Milestone { size_t end; cudaEvent_t ev; };
  std::vector<Milestone> marks;
  {
    size_t topo_end = 0, nodes_end = 0;
    std::vector<size_t> tree_end(ctx->ev_tree.size(), 0);
    for (const CopyJob& j : jobs) {
      const size_t e = j.dst_off + j.bytes;
      if (j.group == 0) topo_end = std::max(topo_end, e);
      if (j.group <= 1) nodes_end = std::max(nodes_end, e);
      if (j.group == 2 && j.tree >= 0 && (size_t)j.tree < tree_end.size()) tree_end[j.tree] = std::max(tree_end[j.tree], e);
    }
    nodes_end = std::max(nodes_end, topo_end);
    marks.push_back({topo_end, ctx->ev_topo});
    marks.push_back({nodes_end, ctx->ev_nodes});
    for (size_t k = 0; k < tree_end.size(); ++k) if (tree_end[k]) marks.push_back({std::max(tree_end[k], nodes_end), ctx->ev_tree[k]});
    std::stable_sort(marks.begin(), marks.end(), [](const Milestone& a, const Milestone& b) { return a.end < b.end; });
  }
  size_t next_mark = 0;
  cudaError_t ce = cudaStreamWaitEvent(cs, ctx->ev_main, 0);
  auto issue_chunk = [&](size_t c) {
    const size_t lo = c * kChunk, hi = std::min(total, lo + kChunk);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(d_base + lo, pinned + lo, hi - lo, cudaMemcpyHostToDevice, cs);
    while (ce == cudaSuccess && next_mark < marks.size() && marks[next_mark].end <= hi) ce = cudaEventRecord(marks[next_mark++].ev, cs);
  };
  auto finish = [&]() {
    while (ce == cudaSuccess && next_mark < marks.size()) ce = cudaEventRecord(marks[next_mark++].ev, cs);
    if (ce == cudaSuccess) ce = cudaEventRecord(ctx->ev_lists, cs);
    *two_phase = ce == cudaSuccess;
    if (ce != cudaSuccess) sync_copy_streams(ctx);
  };
  if (nthreads <= 1) {
    for (size_t c = 0; c < nchunks && ce == cudaSuccess; ++c) {
      fill_chunk(c);
      issue_chunk(c);
    }
    finish();
  } else {
    std::vector<std::atomic<int>> done(nchunks);
    for (auto& d : done) d.store(0, std::memory_order_relaxed);
    std::atomic<size_t> next{0};
    auto worker = [&]() {
      for (;;) {
        const size_t c = next.fetch_add(1, std::memory_order_relaxed);
        if (c >= nchunks) return;
        fill_chunk(c);
        done[c].store(1, std::memory_order_release);
      }
    };
    std::vector<std::thread> pool;
    for (size_t i = 1; i < nthreads; ++i) pool.emplace_back(worker);
    for (size_t c = 0; c < nchunks; ++c) {
      while (!done[c].load(std::memory_order_acquire)) {
        // help out instead of spinning
        const size_t h = next.fetch_add(1, std::memory_order_relaxed);
        if (h < nchunks) { fill_chunk(h); done[h].store(1, std::memory_order_release); } else std::this_thread::yield();
      }
      issue_chunk(c);
    }
    for (auto& th : pool) th.join();
    finish();
  }
  return check_cuda(ctx, ce, "H2D staged upload");
}

int flatten_status_to_error(dphy_ctx* ctx, uint32_t bits) {
  if (bits & kFlattenErrTopology) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "tree topology is not a binary tree rooted at `root`");
  if (bits & kFlattenErrOffsets) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "CSR offsets are not monotone");
  if (bits & kFlattenErrMutSite) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "mutation site out of range");
  if (bits & kFlattenErrMissation) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "Missation out of range");
  if (bits & kFlattenErrMutState) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "mutation state not in ACGT");
  if (bits & kFlattenErrFsState) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "missation from-state not in ACGT");
  if (bits & kFlattenErrTimes) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "a node is earlier than its parent");
  if (bits & kFlattenErrFswRange) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "more than 32,767 from-state overrides of one state on one branch");
  return DPHY_OK;
}

}  // namespace

static int forest_upload_impl(dphy_ctx* ctx, int32_t num_trees, const dphy_emat_host* trees, const TreeTotals* totals, const int32_t* sites_index,
                              int32_t num_sites_tables, dphy_sites* const* sites, dphy_forest** out, const dphy_forest* order_from = nullptr) {
  if (!ctx || !out || num_trees < 0 || (num_trees > 0 && (!trees || !sites)) || num_sites_tables <= 0) return DPHY_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  cudaSetDevice(ctx->device);
  auto tot_m = [&](int k) -> int64_t { return totals ? totals[k].m : trees[k].mut_off[trees[k].num_nodes]; };
  auto tot_iv = [&](int k) -> int64_t { return totals ? totals[k].iv : trees[k].miss_off[trees[k].num_nodes]; };
  auto tot_fs = [&](int k) -> int64_t { return totals ? totals[k].fs : trees[k].fs_off[trees[k].num_nodes]; };
  auto tot_root_m = [&](int k) -> int64_t { return totals ? totals[k].root_m : trees[k].mut_off[trees[k].root + 1] - trees[k].mut_off[trees[k].root]; };
  int64_t N = 0, M = 0, I = 0, F = 0, tiles = 0, ctiles = 0;
  int max_tree_nodes = 0;
  for (int k = 0; k < num_trees; ++k) {
    const auto& e = trees[k];
    if (e.num_nodes <= 0) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "empty tree");
    if (e.root < 0 || e.root >= e.num_nodes) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "root out of range");
    const int si = sites_index ? sites_index[k] : 0;
    if (si < 0 || si >= num_sites_tables) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "sites_index out of range");
    const int n = e.num_nodes;
    if (tot_m(k) < 0 || tot_iv(k) < 0 || tot_fs(k) < 0 || tot_root_m(k) < 0)
      return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "CSR offsets are not monotone");
    N += n; M += tot_m(k); I += tot_iv(k); F += tot_fs(k);
    tiles += (n + kTile - 1) / kTile;
    ctiles += (n + kLgTile - 1) / kLgTile;
    max_tree_nodes = std::max(max_tree_nodes, n);
  }
  if (N > std::numeric_limits<int32_t>::max() / 4 || M > std::numeric_limits<int32_t>::max() / 2 ||
      I > std::numeric_limits<int32_t>::max() / 2 || F > std::numeric_limits<int32_t>::max() / 2)
    return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "forest too large for 32-bit positions");
  int maxP = 1;
  for (int i = 0; i < num_sites_tables; ++i) {
    if (!sites[i]) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "null sites table");
    maxP = std::max(maxP, sites[i]->P);
  }
  const int fsw_stride = 4 * maxP;

  std::unique_ptr<dphy_forest> fo(new (std::nothrow) dphy_forest());
  if (!fo) return DPHY_ERR_OUT_OF_MEMORY;
  fo->total_muts = M; fo->total_ivls = I; fo->total_fs = F;
  fo->sites.assign(sites, sites + num_sites_tables);
  fo->sites_version.resize(num_sites_tables);
  fo->tree_muts.resize(num_trees); fo->tree_fs.resize(num_trees); fo->tree_max_depth.assign(num_trees, 0);
  fo->trees.resize(num_trees);

  // ---- the resident forest slab --------------------------------------------------------------------------------------
  Slab slab;
  const int b_trees = slab.reserve(sizeof(TreeDev) * num_trees);
  const int b_sites = slab.reserve(sizeof(SitesDev) * num_sites_tables);
  const int b_tile_tree = slab.reserve(sizeof(int32_t) * tiles);
  const int b_ctiles = slab.reserve(sizeof(CTileDesc) * ctiles);
  const int b_corder = slab.reserve(sizeof(int32_t) * ctiles);
  const size_t header_bytes = slab.total;
  const int b_node_id = slab.reserve(sizeof(int32_t) * N), b_parent = slab.reserve(sizeof(int32_t) * N);
  const int b_depth = slab.reserve(sizeof(int32_t) * N), b_size = slab.reserve(sizeof(int32_t) * N);
  const int b_post = slab.reserve(sizeof(int32_t) * N), b_pos = slab.reserve(sizeof(int32_t) * N);
  const int b_t = slab.reserve(sizeof(double) * N);
  const int b_moff = slab.reserve(sizeof(int32_t) * (N + 1)), b_msite = slab.reserve(sizeof(int32_t) * M + 64);
  const int b_mft = slab.reserve(M + 64), b_mt = slab.reserve(sizeof(double) * M + 64);
  const int b_ioff = slab.reserve(sizeof(int32_t) * (N + 1)), b_is = slab.reserve(sizeof(int2) * I + 64);
  const int b_foff = slab.reserve(sizeof(int32_t) * (N + 1)), b_fsite = slab.reserve(sizeof(int32_t) * F + 64), b_ffrom = slab.reserve(F + 64);
  const int b_fsw = slab.reserve(sizeof(int16_t) * (size_t)fsw_stride * N + 64);
  const int b_cnt = slab.reserve(sizeof(int32_t) * (size_t)fsw_stride * N + 64);
  // outputs + workspaces
  const int b_lambda = slab.reserve(sizeof(double) * N), b_nsmn = slab.reserve(sizeof(int32_t) * N);
  const int b_strad = slab.reserve(sizeof(int32_t) * 2 * N), b_sdd = slab.reserve(sizeof(double) * N), b_sdn = slab.reserve(sizeof(int32_t) * N);
  const int b_tout = slab.reserve(sizeof(double) * 4 * num_trees), b_tiout = slab.reserve(sizeof(int32_t) * 20 * num_trees);
  const int b_tagg = slab.reserve(sizeof(double) * tiles), b_tiagg = slab.reserve(sizeof(int32_t) * tiles);
  const int b_tpart = slab.reserve(sizeof(double) * 2 * tiles), b_tipart = slab.reserve(sizeof(int32_t) * 17 * tiles);
  const int b_tflag = slab.reserve(sizeof(uint32_t) * tiles);

  // ---- the temporary block: raw host-order arrays + flatten workspaces -------------------------------------------------------
  Slab tmp;
  const int r_raw = tmp.reserve(sizeof(RawTreeDev) * num_trees);
  struct RawIds { int parent, c0, c1, t, moff, msite, mfrom, mto, mt, ioff, is, ie, foff, fsite, ffrom; };
  std::vector<RawIds> rid(num_trees);
  // group-major: every tree's topology arrays first, then the node times + CSR offsets, then the lists tree by tree -- the order
  // in which the flatten stages need them, so that a staged (in destination order) upload releases the stages early too
  for (int k = 0; k < num_trees; ++k) {
    const size_t n = trees[k].num_nodes;
    RawIds& r = rid[k];
    r.parent = tmp.reserve(4 * n); r.c0 = tmp.reserve(4 * n); r.c1 = tmp.reserve(4 * n);
  }
  for (int k = 0; k < num_trees; ++k) {
    const size_t n = trees[k].num_nodes;
    RawIds& r = rid[k];
    r.t = tmp.reserve(8 * n); r.moff = tmp.reserve(4 * (n + 1)); r.ioff = tmp.reserve(4 * (n + 1)); r.foff = tmp.reserve(4 * (n + 1));
  }
  for (int k = 0; k < num_trees; ++k) {
    const size_t m = tot_m(k), iv = tot_iv(k), fs = tot_fs(k);
    RawIds& r = rid[k];
    r.msite = tmp.reserve(4 * m); r.mfrom = tmp.reserve(m); r.mto = tmp.reserve(m); r.mt = tmp.reserve(8 * m);
    r.is = tmp.reserve(4 * iv); r.ie = tmp.reserve(4 * iv);
    r.fsite = tmp.reserve(4 * fs); r.ffrom = tmp.reserve(fs);
  }
  const size_t raw_upload_bytes = tmp.total;
  // the raw (host-order) arrays stay resident next to the flattened forest: dphy_forest_apply_rows patches them on the device and
  // re-flattens from there, so an edited tree never crosses PCIe again.  The flatten workspaces live in their own block, freed below.
  Slab work;
  // the Euler-tour arcs (two ping-pong buffers of 2N int4) are dead once the node records are scattered: the count scan's
  // post-order prefix (N rows of fsw_stride int32) reuses their block
  const int w_arcs = work.reserve(std::max(sizeof(int4) * 4 * N, sizeof(int32_t) * (size_t)fsw_stride * N));
  const int64_t scan_tiles = (N + 1023) / 1024;
  const int w_scan = work.reserve(sizeof(int32_t) * 3 * scan_tiles);
  const int w_cnttot = work.reserve(sizeof(uint4) * 2 * (fsw_stride / 4) * scan_tiles);
  const int w_status = work.reserve(sizeof(uint32_t) * 2 + sizeof(int32_t) * num_trees);
  const int w_jobs = work.reserve(sizeof(DeviceCopyJob) * ((size_t)num_trees * 15 + 1));     // device-resident sources only (see below)

  DevBlock dblk(ctx->stream), tblk(ctx->stream), wblk(ctx->stream);
  if (!dblk.alloc(slab.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(forest)");
  if (!tblk.alloc(tmp.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(forest raw arrays)");
  if (!wblk.alloc(work.total)) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "cudaMallocAsync(forest workspace)");
  char* dbase = dblk.p; char* tbase = tblk.p; char* wbase = wblk.p;
  fo->bytes = slab.total;
  if (ensure_copy_stream(ctx) != DPHY_OK || cudaEventRecord(ctx->ev_main, ctx->stream) != cudaSuccess)
    return set_error(ctx, DPHY_ERR_CUDA, "upload: copy stream / event");

  PinnedStage pin(ctx, header_bytes + raw_upload_bytes);
  if (pin.status != DPHY_OK) return pin.status;
  int st = DPHY_OK;
  char* hb = pin.p;                            // [header | raw]
  char* hraw = hb + header_bytes;

  // ---- host side: only the per-tree / per-tile descriptors; the arrays are streamed verbatim ---------------------------
  auto* h_trees = slab.at<TreeDev>(hb, b_trees);
  auto* h_sites = slab.at<SitesDev>(hb, b_sites);
  auto* h_tile_tree = slab.at<int32_t>(hb, b_tile_tree);
  auto* h_ctiles = slab.at<CTileDesc>(hb, b_ctiles);
  auto* h_corder = slab.at<int32_t>(hb, b_corder);
  auto* h_raw = tmp.at<RawTreeDev>(hraw, r_raw);
  for (int i = 0; i < num_sites_tables; ++i) { h_sites[i] = sites[i]->h; fo->sites_version[i] = sites[i]->version; }
  std::vector<CopyJob> jobs;
  jobs.reserve((size_t)num_trees * 15 + 1);
  jobs.push_back({tmp.blocks[r_raw].off, h_raw, sizeof(RawTreeDev) * (size_t)num_trees, 0, -1});   // written in place below
  int32_t base = 0, tile_pos = 0, ctile_pos = 0;
  for (int k = 0; k < num_trees; ++k) {
    const auto& e = trees[k];
    const int n = e.num_nodes;
    const size_t m = tot_m(k), iv = tot_iv(k), fs = tot_fs(k);
    TreeDev& T = fo->trees[k];
    T.node_base = base; T.num_nodes = n; T.sites_id = sites_index ? sites_index[k] : 0; T.first_tile = tile_pos;
    T.num_tiles = (n + kTile - 1) / kTile; T.includes_run_root = e.includes_run_root; T.root_id = e.root; T.pad = 0;
    for (int j = 0; j < T.num_tiles; ++j) h_tile_tree[tile_pos++] = k;
    T.first_ctile = ctile_pos; T.num_ctiles = (n + kLgTile - 1) / kLgTile;
    for (int j = 0; j < T.num_ctiles; ++j) {
      CTileDesc& d = h_ctiles[ctile_pos++];
      std::memset(&d, 0, sizeof(d));
      d.tile_start = base + j * kLgTile; d.n_act = std::min(kLgTile, n - j * kLgTile); d.node_base = base; d.sites_id = T.sites_id;
    }
    h_trees[k] = T;
    fo->tree_muts[k] = (int64_t)m; fo->tree_fs[k] = (int64_t)fs;
    const RawIds& r = rid[k];
    RawTreeDev& R = h_raw[k];
    R.parent = tmp.at<int32_t>(tbase, r.parent); R.child0 = tmp.at<int32_t>(tbase, r.c0); R.child1 = tmp.at<int32_t>(tbase, r.c1);
    R.t = tmp.at<double>(tbase, r.t);
    R.mut_off = tmp.at<int32_t>(tbase, r.moff); R.mut_site = tmp.at<int32_t>(tbase, r.msite);
    R.mut_from = tmp.at<uint8_t>(tbase, r.mfrom); R.mut_to = tmp.at<uint8_t>(tbase, r.mto); R.mut_t = tmp.at<double>(tbase, r.mt);
    R.miss_off = tmp.at<int32_t>(tbase, r.ioff); R.miss_start = tmp.at<int32_t>(tbase, r.is); R.miss_end = tmp.at<int32_t>(tbase, r.ie);
    R.fs_off = tmp.at<int32_t>(tbase, r.foff); R.fs_site = tmp.at<int32_t>(tbase, r.fsite); R.fs_from = tmp.at<uint8_t>(tbase, r.ffrom);
    R.root = e.root; R.num_nodes = n; R.num_muts = (int32_t)m; R.num_ivls = (int32_t)iv; R.num_fs = (int32_t)fs; R.pad = 0;
    auto add = [&](int id, const void* src, size_t bytes, int group = 2) { if (bytes) jobs.push_back({tmp.blocks[id].off, src, bytes, group, k}); };
    add(r.parent, e.parent, 4 * (size_t)n, 0); add(r.c0, e.child0, 4 * (size_t)n, 0); add(r.c1, e.child1, 4 * (size_t)n, 0); add(r.t, e.t, 8 * (size_t)n, 1);
    add(r.moff, e.mut_off, 4 * ((size_t)n + 1), 1); add(r.msite, e.mut_site, 4 * m); add(r.mfrom, e.mut_from, m); add(r.mto, e.mut_to, m); add(r.mt, e.mut_t, 8 * m);
    add(r.ioff, e.miss_off, 4 * ((size_t)n + 1), 1); add(r.is, e.miss_start, 4 * iv); add(r.ie, e.miss_end, 4 * iv);
    add(r.foff, e.fs_off, 4 * ((size_t)n + 1), 1); add(r.fsite, e.fs_site, 4 * fs); add(r.ffrom, e.fs_from, fs);
    base += n;
  }

  // launch order of the general log-G tile kernel: full tiles first, every tree's partly filled last tile at the end (fullest
  // first), so that the last wave of a many-small-trees forest is made of the cheap tiles
  {
    int w = 0;
    for (int j = 0; j < (int)ctiles; ++j) if (h_ctiles[j].n_act == kLgTile) h_corder[w++] = j;
    const int first_partial = w;
    for (int j = 0; j < (int)ctiles; ++j) if (h_ctiles[j].n_act != kLgTile) h_corder[w++] = j;
    std::stable_sort(h_corder + first_partial, h_corder + w, [&](int a, int b) { return h_ctiles[a].n_act > h_ctiles[b].n_act; });
  }
  cudaError_t ce = cudaMemcpyAsync(dbase, hb, header_bytes, cudaMemcpyHostToDevice, ctx->stream);
  if (ce == cudaSuccess) ce = cudaMemsetAsync(dbase + header_bytes, 0, slab.total - header_bytes, ctx->stream);
  if (ce == cudaSuccess) ce = cudaMemsetAsync(wbase + work.blocks[w_status].off, 0, work.blocks[w_status].bytes, ctx->stream);
  if (ce != cudaSuccess) return check_cuda(ctx, ce, "H2D forest header");
  // the RawTreeDev records were written straight into the pinned slab above; everything in [0, raw_upload_bytes) not
  // covered by a job (those records, alignment gaps) is copied as it lies
  while ((int)ctx->ev_tree.size() < num_trees) {
    cudaEvent_t e = nullptr;
    if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return set_error(ctx, DPHY_ERR_CUDA, "cudaEventCreate");
    ctx->ev_tree.push_back(e);
  }
  std::vector<char> tree_has_lists(num_trees, 0);
  for (const CopyJob& j : jobs) if (j.group == 2 && j.tree >= 0) tree_has_lists[j.tree] = 1;
  bool two_phase = false;
  if (totals) {
    // device-resident sources (dphy_forest_apply_rows): ONE kernel copies every array (the copy-stream path above costs a driver
    // call and an event or two per array -- 240 arrays for 16 trees, more host time than all the kernels of the rebuild)
    DeviceCopyJob* hj = reinterpret_cast<DeviceCopyJob*>(hraw + align_up(tmp.blocks[r_raw].off + sizeof(RawTreeDev) * (size_t)num_trees));
    int nj = 0;
    size_t max_bytes = 1;
    cudaError_t ce2 = cudaSuccess;
    for (const CopyJob& j : jobs) {
      if (j.tree < 0) { ce2 = cudaMemcpyAsync(tbase + j.dst_off, j.src, j.bytes, cudaMemcpyHostToDevice, ctx->stream); continue; }   // the per-tree records
      hj[nj++] = DeviceCopyJob{tbase + j.dst_off, static_cast<const char*>(j.src), j.bytes};
      max_bytes = std::max(max_bytes, j.bytes);
    }
    DeviceCopyJob* dj = work.at<DeviceCopyJob>(wbase, w_jobs);
    if (ce2 == cudaSuccess && nj > 0) ce2 = cudaMemcpyAsync(dj, hj, sizeof(DeviceCopyJob) * nj, cudaMemcpyHostToDevice, ctx->stream);
    if (ce2 == cudaSuccess && nj > 0) st = launch_device_copies(ctx, dj, nj, max_bytes);
    else st = check_cuda(ctx, ce2, "device copy jobs");
  } else {
    st = staged_upload(ctx, hraw, jobs, tbase, raw_upload_bytes, &two_phase);
  }
  if (!two_phase) pin.reset();           // (two-phase: once the copy streams are joined below)
  if (st != DPHY_OK) return st;

  ForestDev& h = fo->h;
  h.num_trees = num_trees; h.num_nodes = (int32_t)N; h.num_tiles = (int32_t)tiles; h.num_sites_tables = num_sites_tables;
  h.trees = slab.at<TreeDev>(dbase, b_trees); h.sites = slab.at<SitesDev>(dbase, b_sites);
  h.tile_tree = slab.at<int32_t>(dbase, b_tile_tree);
  h.num_ctiles = (int32_t)ctiles; h.pad0 = 0; h.ctiles = slab.at<CTileDesc>(dbase, b_ctiles);
  h.node_id = slab.at<int32_t>(dbase, b_node_id); h.parent_pos = slab.at<int32_t>(dbase, b_parent);
  h.depth = slab.at<int32_t>(dbase, b_depth); h.subtree_size = slab.at<int32_t>(dbase, b_size);
  h.post_node = slab.at<int32_t>(dbase, b_post); h.pos_of_node = slab.at<int32_t>(dbase, b_pos);
  h.t = slab.at<double>(dbase, b_t);
  h.mut_off = slab.at<int32_t>(dbase, b_moff); h.mut_site = slab.at<int32_t>(dbase, b_msite);
  h.mut_code = slab.at<uint8_t>(dbase, b_mft); h.mut_t = slab.at<double>(dbase, b_mt);
  h.miss_off = slab.at<int32_t>(dbase, b_ioff); h.miss_se = slab.at<int2>(dbase, b_is);
  h.fs_off = slab.at<int32_t>(dbase, b_foff); h.fs_site = slab.at<int32_t>(dbase, b_fsite); h.fs_code = slab.at<uint8_t>(dbase, b_ffrom);
  h.fsw = slab.at<int16_t>(dbase, b_fsw); h.fsw_stride = fsw_stride; h.pad1 = 0;
  h.C = slab.at<int32_t>(dbase, b_cnt);
  fo->d_lambda = slab.at<double>(dbase, b_lambda); fo->d_nsmn = slab.at<int32_t>(dbase, b_nsmn);
  fo->d_tree_out = slab.at<double>(dbase, b_tout); fo->d_tree_iout = slab.at<int32_t>(dbase, b_tiout);
  fo->d_tile_agg = slab.at<double>(dbase, b_tagg); fo->d_tile_iagg = slab.at<int32_t>(dbase, b_tiagg);
  fo->d_tile_part = slab.at<double>(dbase, b_tpart); fo->d_tile_ipart = slab.at<int32_t>(dbase, b_tipart);
  fo->d_tile_flag = slab.at<uint32_t>(dbase, b_tflag);
  fo->d_ctile_order = slab.at<int32_t>(dbase, b_corder);
  fo->d_strad_list = slab.at<int32_t>(dbase, b_strad); fo->d_sd_delta = slab.at<double>(dbase, b_sdd); fo->d_sd_n = slab.at<int32_t>(dbase, b_sdn);

  // ---- device side: Euler tour + list ranking -> DFS order; CSR offsets; lists ------------------------------------------
  FlattenParams P{};
  P.trees = h.trees; P.sites = h.sites; P.tile_tree = h.tile_tree; P.raw = tmp.at<RawTreeDev>(tbase, r_raw);
  P.arcs[0] = work.at<int4>(wbase, w_arcs); P.arcs[1] = P.arcs[0] + 2 * N;
  P.scan_tiles = work.at<int32_t>(wbase, w_scan);
  P.status = work.at<uint32_t>(wbase, w_status); P.max_depth = reinterpret_cast<int32_t*>(P.status + 2);
  P.strad_list = fo->d_strad_list;
  P.ctiles = const_cast<CTileDesc*>(h.ctiles); P.num_ctiles = (int32_t)ctiles;
  P.num_nodes = (int32_t)N; P.total_muts = (int32_t)M; P.total_ivls = (int32_t)I; P.total_fs = (int32_t)F;
  P.node_id = const_cast<int32_t*>(h.node_id); P.parent_pos = const_cast<int32_t*>(h.parent_pos);
  P.depth = const_cast<int32_t*>(h.depth); P.subtree_size = const_cast<int32_t*>(h.subtree_size);
  P.post_node = const_cast<int32_t*>(h.post_node); P.pos_of_node = const_cast<int32_t*>(h.pos_of_node);
  P.t = h.t;
  P.mut_off = const_cast<int32_t*>(h.mut_off); P.mut_site = const_cast<int32_t*>(h.mut_site);
  P.mut_code = const_cast<uint8_t*>(h.mut_code); P.mut_t = h.mut_t;
  P.miss_off = const_cast<int32_t*>(h.miss_off); P.miss_se = const_cast<int2*>(h.miss_se);
  P.fs_off = const_cast<int32_t*>(h.fs_off); P.fs_site = const_cast<int32_t*>(h.fs_site); P.fs_code = const_cast<uint8_t*>(h.fs_code);
  P.fsw = const_cast<int16_t*>(h.fsw); P.fsw_stride = fsw_stride;
  P.C = const_cast<int32_t*>(h.C);
  P.cnt_y = work.at<int32_t>(wbase, w_arcs); P.cnt_tot = work.at<uint4>(wbase, w_cnttot);
  if (order_from) {
    P.old_pos_of_node = order_from->h.pos_of_node; P.old_depth = order_from->h.depth; P.old_subtree_size = order_from->h.subtree_size;
    P.old_parent_pos = order_from->h.parent_pos;
  }
  if (two_phase) {
    // Euler-tour ranking as soon as the topology arrays have landed; the rest once the lists have
    ce = cudaStreamWaitEvent(ctx->stream, ctx->ev_topo, 0);
    if (ce != cudaSuccess) return check_cuda(ctx, ce, "wait topology upload");
    st = launch_flatten(ctx, P, (int)tiles, max_tree_nodes, 0);
    if (st != DPHY_OK) { sync_copy_streams(ctx); return st; }
    ce = cudaStreamWaitEvent(ctx->stream, ctx->ev_nodes, 0);
    if (ce != cudaSuccess) { sync_copy_streams(ctx); return check_cuda(ctx, ce, "wait node upload"); }
    st = launch_flatten(ctx, P, (int)tiles, max_tree_nodes, 1);
    if (st != DPHY_OK) { sync_copy_streams(ctx); return st; }
    // lists: each tree is gathered and folded as soon as its own arrays have landed, while the next trees' are still in flight
    for (int k = 0; k < num_trees && st == DPHY_OK; ++k) {
      if (tree_has_lists[k]) {
        ce = cudaStreamWaitEvent(ctx->stream, ctx->ev_tree[k], 0);
        if (ce != cudaSuccess) { st = check_cuda(ctx, ce, "wait list upload"); break; }
      }
      st = launch_flatten_lists(ctx, P, fo->trees[k].first_tile, fo->trees[k].num_tiles);
    }
    if (st == DPHY_OK) {
      ce = cudaStreamWaitEvent(ctx->stream, ctx->ev_lists, 0);
      if (ce != cudaSuccess) st = check_cuda(ctx, ce, "wait list upload");
    }
    if (st != DPHY_OK) { sync_copy_streams(ctx); return st; }
    pin.reset();
    st = launch_flatten_finish(ctx, P);
  } else {
    st = launch_flatten(ctx, P, (int)tiles, max_tree_nodes);
  }
  if (st != DPHY_OK) return st;
  std::vector<int32_t> status(2 + num_trees, 0);
  ce = cudaMemcpyAsync(status.data(), P.status, sizeof(int32_t) * status.size(), cudaMemcpyDeviceToHost, ctx->stream);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
  if (ce != cudaSuccess) return check_cuda(ctx, ce, "forest flatten");
  st = flatten_status_to_error(ctx, (uint32_t)status[0]);
  if (st != DPHY_OK) return st;
  for (int k = 0; k < num_trees; ++k) fo->tree_max_depth[k] = status[2 + k];
  fo->num_strad = status[1];
  wblk.reset();
  fo->bytes += tmp.total;
  fo->raw.assign(h_raw, h_raw + num_trees);          // device pointers of every tree's host-order arrays
  fo->sites_index.resize(num_trees);
  for (int k = 0; k < num_trees; ++k) fo->sites_index[k] = sites_index ? sites_index[k] : 0;
  // first evaluation.  Forests whose site rates are uniform take the folded schedule; the structure-only outputs (nsmn, the
  // num_muts tallies) then come from a general pass the first time a getter asks for them (ensure_struct_outputs)
  st = launch_log_G(ctx, fo.get());
  if (st != DPHY_OK) { cudaStreamSynchronize(ctx->stream); return st; }
  fo->allocs.push_back(dblk.release());
  fo->allocs.push_back(tblk.release());              // the raw arrays stay (freed with the forest)
  fo->evaluated = true;         // that pass is a complete evaluation under the current evo model
  fo->eval_version.resize(fo->sites.size());
  for (size_t i = 0; i < fo->sites.size(); ++i) fo->eval_version[i] = fo->sites[i]->version;
  *out = fo.release();
  return DPHY_OK;
}

int dphy_forest_upload(dphy_ctx* ctx, int32_t num_trees, const dphy_emat_host* trees, const int32_t* sites_index,
                       int32_t num_sites_tables, dphy_sites* const* sites, dphy_forest** out) {
  return forest_upload_impl(ctx, num_trees, trees, nullptr, sites_index, num_sites_tables, sites, out);
}

}  // extern "C"

// A new forest from host-order arrays that already lie on the device (dphy_forest_upload_api_trees): the upload path with device sources.
int dphy::forest_from_device_arrays(dphy_ctx* ctx, int32_t num_trees, const dphy_emat_host* views, const TreeTotals* totals, const int32_t* sites_index,
                                    int32_t num_sites_tables, dphy_sites* const* sites, dphy_forest** out) {
  return forest_upload_impl(ctx, num_trees, views, totals, sites_index, num_sites_tables, sites, out);
}

// Re-flatten `fo` from device-resident host-order arrays (dphy_forest_apply_rows): a fresh forest is built by the upload path with
// device sources, then swapped into the caller's handle; the old contents are released stream-ordered.  On failure `fo` is untouched.
int dphy::rebuild_forest_from_device(dphy_ctx* ctx, dphy_forest* fo, const dphy_emat_host* trees, const TreeTotals* totals, bool same_links) {
  dphy_forest* fresh = nullptr;
  const std::vector<dphy_sites*> sites = fo->sites;
  const std::vector<int32_t> si = fo->sites_index;
  int st = forest_upload_impl(ctx, fo->h.num_trees, trees, totals, si.data(), (int32_t)sites.size(), sites.data(), &fresh, same_links ? fo : nullptr);
  if (st != DPHY_OK) return st;
  fresh->cnt_mut = std::move(fo->cnt_mut); fresh->cnt_miss = std::move(fo->cnt_miss); fresh->cnt_fs = std::move(fo->cnt_fs);
  std::swap(*fo, *fresh);
  dphy_forest_destroy(ctx, fresh);
  return DPHY_OK;
}

extern "C" {

void dphy_forest_destroy(dphy_ctx* ctx, dphy_forest* fo) {
  if (!fo) return;
  if (ctx) {
    dphy_ctx_join_side_streams(ctx);      // the tail of an SPR batch may still be reading this forest
    // blocks parked by destroyed SPR batches (dphy_ctx::spr_blocks) go back to the pool with the forest they were sized for
    for (auto& blk : ctx->spr_blocks) {
      if (blk.ev) { cudaStreamWaitEvent(ctx->stream, blk.ev, 0); cudaEventDestroy(blk.ev); }
      cudaFreeAsync(blk.ptr, ctx->stream);
    }
    ctx->spr_blocks.clear();
  }
  if (ctx) {
    cudaSetDevice(ctx->device);
    for (void* p : fo->allocs) cudaFreeAsync(p, ctx->stream);   // stream-ordered: returns to the pool, no device sync
  } else {
    for (void* p : fo->allocs) cudaFree(p);
  }
  delete fo;
}

int64_t dphy_forest_num_nodes(const dphy_forest* fo) { return fo ? fo->h.num_nodes : 0; }
int64_t dphy_forest_device_bytes(const dphy_forest* fo) { return fo ? (int64_t)fo->bytes : 0; }

int64_t dphy_forest_log_G_algorithmic_bytes(const dphy_forest* fo) {
  if (!fo) return 0;
  // SURVEY.md section 8(d): N*(4 parent + 8 t + 4+4+4 CSR offsets) + M*(4 site + 1 from|to + 8 t) + M*8 (nu_l gather)
  //                         + I*(4+4) + I*16 (two cum_Q gathers) + F*(4+1) + F*8 + N*8 (lambda_i written once) + 8/tree
  const int64_t N = fo->h.num_nodes, M = fo->total_muts, I = fo->total_ivls, F = fo->total_fs;
  int64_t nu_bytes = 0;   // "[nu on: M*8 + F*8]" -- only trees whose site table has site-rate heterogeneity
  for (size_t k = 0; k < fo->trees.size(); ++k)
    if (!fo->sites[fo->trees[k].sites_id]->h.nu_uniform) nu_bytes += 8 * (fo->tree_muts[k] + fo->tree_fs[k]);
  return N * 24 + M * 13 + I * 8 + I * 16 + F * 5 + nu_bytes + N * 8 + 8 * (int64_t)fo->h.num_trees;
}

int dphy_forest_set_node_times(dphy_ctx* ctx, dphy_forest* fo, int32_t tree, int32_t count, const int32_t* nodes, const double* t) {
  if (ctx) dphy_ctx_join_side_streams(ctx);        // the tail of an SPR batch may still be reading the node times
  if (!ctx || !fo || tree < 0 || tree >= fo->h.num_trees || count < 0 || (count > 0 && (!nodes || !t))) return DPHY_ERR_INVALID_ARGUMENT;
  if (count == 0) return DPHY_OK;
  // the tree's dated placement index is stale from here on, also when the checks below fail after some times were written
  if (fo->times_version.size() != fo->trees.size()) fo->times_version.assign(fo->trees.size(), 0);
  ++fo->times_version[tree];
  cudaSetDevice(ctx->device);
  const size_t mark = ctx->arena.mark();
  int32_t* d_nodes = (int32_t*)ctx->arena.alloc(sizeof(int32_t) * count);
  double* d_vals = (double*)ctx->arena.alloc(sizeof(double) * count);
  uint32_t* d_status = (uint32_t*)ctx->arena.alloc(sizeof(uint32_t));
  if (!d_nodes || !d_vals || !d_status) { ctx->arena.release(mark); return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "arena exhausted (set_node_times)"); }
  uint32_t status = 0;
  int st = check_cuda(ctx, cudaMemcpyAsync(d_nodes, nodes, sizeof(int32_t) * count, cudaMemcpyHostToDevice, ctx->stream), "H2D");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaMemcpyAsync(d_vals, t, sizeof(double) * count, cudaMemcpyHostToDevice, ctx->stream), "H2D");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaMemsetAsync(d_status, 0, sizeof(uint32_t), ctx->stream), "memset");
  if (st == DPHY_OK) st = launch_set_node_times(ctx, fo, tree, d_nodes, d_vals, count, d_status);
  if (st == DPHY_OK) st = launch_raw_set_node_times(ctx, fo, tree, d_nodes, d_vals, count);   // the resident host-order copy follows
  if (st == DPHY_OK) st = check_cuda(ctx, cudaMemcpyAsync(&status, d_status, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream), "D2H");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "set_node_times");
  ctx->arena.release(mark);
  fo->evaluated = false;
  if (st == DPHY_OK && (status & 1u)) return set_error(ctx, DPHY_ERR_OUT_OF_RANGE, "node out of range");
  if (st == DPHY_OK && (status & 2u)) return set_error(ctx, DPHY_ERR_INVALID_ARGUMENT, "a displaced node is no longer between its parent and its children");
  return st;
}

// ---- log G ----------------------------------------------------------------------------------------------------------
int dphy_forest_eval_log_G(dphy_ctx* ctx, dphy_forest* fo) {
  if (!ctx || !fo) return DPHY_ERR_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  int st = launch_log_G(ctx, fo);
  if (st == DPHY_OK) {
    fo->evaluated = true;
    fo->eval_version.resize(fo->sites.size());
    for (size_t i = 0; i < fo->sites.size(); ++i) fo->eval_version[i] = fo->sites[i]->version;
  }
  return st;
}

// nsmn and the num_muts tallies depend on the tree alone and are produced by the general schedule only: run it once if the
// forest has so far been evaluated by the folded schedule alone (it also re-derives everything else, consistently)
static int ensure_struct_outputs(dphy_ctx* ctx, dphy_forest* fo) {
  if (fo->struct_valid) return DPHY_OK;
  int st = launch_log_G_general(ctx, fo);
  if (st == DPHY_OK) {
    fo->evaluated = true;
    fo->eval_version.resize(fo->sites.size());
    for (size_t i = 0; i < fo->sites.size(); ++i) fo->eval_version[i] = fo->sites[i]->version;
  }
  return st;
}

static int fetch_tree_outputs(dphy_ctx* ctx, dphy_forest* fo, std::vector<double>& dout, std::vector<int32_t>* iout) {
  if (iout) { int st = ensure_struct_outputs(ctx, fo); if (st != DPHY_OK) return st; }
  if (!fo->eval_current()) { int st = dphy_forest_eval_log_G(ctx, fo); if (st != DPHY_OK) return st; }
  const int T = fo->h.num_trees;
  dout.resize((size_t)T * 4);
  DPHY_CUDA(ctx, cudaMemcpyAsync(dout.data(), fo->d_tree_out, sizeof(double) * 4 * T, cudaMemcpyDeviceToHost, ctx->stream));
  if (iout) {
    iout->resize((size_t)T * 20);
    DPHY_CUDA(ctx, cudaMemcpyAsync(iout->data(), fo->d_tree_iout, sizeof(int32_t) * 20 * T, cudaMemcpyDeviceToHost, ctx->stream));
  }
  return check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "log G D2H");
}

int dphy_forest_get_log_G(dphy_ctx* ctx, dphy_forest* fo, double* log_root_prior, double* log_G_below_root, double* log_G) {
  if (!ctx || !fo) return DPHY_ERR_INVALID_ARGUMENT;
  std::vector<double> d;
  int st = fetch_tree_outputs(ctx, fo, d, nullptr);
  if (st != DPHY_OK) return st;
  for (int k = 0; k < fo->h.num_trees; ++k) {
    const double rp = d[k * 4 + 0], br = d[k * 4 + 1];
    if (log_root_prior) log_root_prior[k] = rp;
    if (log_G_below_root) log_G_below_root[k] = br;
    if (log_G) log_G[k] = (fo->trees[k].includes_run_root ? rp : 0.0) + br;   // Subrun::calc_cur_log_G
  }
  return DPHY_OK;
}

int dphy_forest_get_lambda_i(dphy_ctx* ctx, dphy_forest* fo, int32_t tree, double* out) {
  if (!ctx || !fo || !out || tree < 0 || tree >= fo->h.num_trees) return DPHY_ERR_INVALID_ARGUMENT;
  if (!fo->eval_current()) { int st = dphy_forest_eval_log_G(ctx, fo); if (st != DPHY_OK) return st; }
  const TreeDev& T = fo->trees[tree];
  const size_t mark = ctx->arena.mark();
  double* tmp = (double*)ctx->arena.alloc(sizeof(double) * T.num_nodes);
  if (!tmp) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "arena exhausted (lambda_i)");
  int st = gather_lambda_host_order(ctx, fo, tree, tmp);
  if (st == DPHY_OK) st = check_cuda(ctx, cudaMemcpyAsync(out, tmp, sizeof(double) * T.num_nodes, cudaMemcpyDeviceToHost, ctx->stream), "lambda_i D2H");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "lambda_i D2H");
  ctx->arena.release(mark);
  return st;
}

int dphy_forest_get_num_sites_missing(dphy_ctx* ctx, dphy_forest* fo, int32_t tree, int32_t* out) {
  if (!ctx || !fo || !out || tree < 0 || tree >= fo->h.num_trees) return DPHY_ERR_INVALID_ARGUMENT;
  { int st = ensure_struct_outputs(ctx, fo); if (st != DPHY_OK) return st; }
  const TreeDev& T = fo->trees[tree];
  const size_t mark = ctx->arena.mark();
  int32_t* tmp = (int32_t*)ctx->arena.alloc(sizeof(int32_t) * T.num_nodes);
  if (!tmp) return set_error(ctx, DPHY_ERR_OUT_OF_MEMORY, "arena exhausted (nsmn)");
  int st = gather_nsmn_host_order(ctx, fo, tree, tmp);
  if (st == DPHY_OK) st = check_cuda(ctx, cudaMemcpyAsync(out, tmp, sizeof(int32_t) * T.num_nodes, cudaMemcpyDeviceToHost, ctx->stream), "nsmn D2H");
  if (st == DPHY_OK) st = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "nsmn D2H");
  ctx->arena.release(mark);
  return st;
}

int dphy_forest_calc_tallies(dphy_ctx* ctx, dphy_forest* fo, dphy_tallies* out) {
  if (!ctx || !fo || !out) return DPHY_ERR_INVALID_ARGUMENT;
  std::vector<double> d; std::vector<int32_t> iv;
  int st = fetch_tree_outputs(ctx, fo, d, &iv);
  if (st != DPHY_OK) return st;
  for (int k = 0; k < fo->h.num_trees; ++k) {
    dphy_tallies& o = out[k];
    o.num_muts = iv[k * 20 + 0]; o.reserved = 0;
    for (int i = 0; i < 16; ++i) o.num_muts_ab[i] = iv[k * 20 + 2 + i];
    o.log_root_prior = fo->trees[k].includes_run_root ? d[k * 4 + 0] : 0.0;
    o.log_G_below_root = d[k * 4 + 1];
    o.T = d[k * 4 + 2];
  }
  return DPHY_OK;
}

int dphy_log_G_host(dphy_ctx* ctx, const dphy_emat_host* tree, const dphy_sites_host* sites, double* log_root_prior,
                    double* log_G_below_root, double* lambda_i) {
  if (!ctx || !tree || !sites) return DPHY_ERR_INVALID_ARGUMENT;
  dphy_sites* s = nullptr; dphy_forest* fo = nullptr;
  int st = dphy_sites_upload(ctx, sites, &s);
  if (st != DPHY_OK) return st;
  int32_t zero = 0;
  st = dphy_forest_upload(ctx, 1, tree, &zero, 1, &s, &fo);
  if (st == DPHY_OK) st = dphy_forest_eval_log_G(ctx, fo);
  if (st == DPHY_OK) st = dphy_forest_get_log_G(ctx, fo, log_root_prior, log_G_below_root, nullptr);
  if (st == DPHY_OK && lambda_i) st = dphy_forest_get_lambda_i(ctx, fo, 0, lambda_i);
  dphy_forest_destroy(ctx, fo);
  dphy_sites_destroy(ctx, s);
  return st;
}

}  // extern "C"
