// device_utils.cuh -- warp/block primitives and memory-ordering helpers shared by the sm_100a kernels.
#ifndef DPHY_DEVICE_UTILS_CUH_
#define DPHY_DEVICE_UTILS_CUH_

#include <cuda_runtime.h>
#include <stdint.h>

namespace dphy {

__device__ __forceinline__ void st_release_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ double ld_cg_f64(const double* p) { return __ldcg(p); }

// Deterministic butterfly reductions (fixed association => bit-reproducible run to run).
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Inclusive warp scans.
__device__ __forceinline__ double warp_scan_incl(double v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    double u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += u;
  }
  return v;
}
__device__ __forceinline__ int warp_scan_incl(int v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += u;
  }
  return v;
}

// Block-wide inclusive scan for blockDim.x == NT (multiple of 32, <= 1024).  `ws` is NT/32 elements of smem.
// Returns the inclusive prefix; *total receives the block total.  Contains two __syncthreads().
template <typename T, int NT>
__device__ __forceinline__ T block_scan_incl(T v, T* ws, T* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int NW = NT / 32;
  T incl = warp_scan_incl(v, lane);
  if (lane == 31) ws[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    T w = lane < NW ? ws[lane] : T(0);
    T wi = warp_scan_incl(w, lane);
    if (lane < NW) ws[lane] = wi;
  }
  __syncthreads();
  T base = warp > 0 ? ws[warp - 1] : T(0);
  *total = ws[NW - 1];
  return incl + base;
}

// Block-wide deterministic sum for blockDim.x == NT.  Result valid in thread 0 (and all of warp 0).
template <typename T, int NT>
__device__ __forceinline__ T block_sum(T v, T* ws) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int NW = NT / 32;
  v = warp_sum(v);
  __syncthreads();          // protect ws against a previous use
  if (lane == 0) ws[warp] = v;
  __syncthreads();
  T r = T(0);
  if (warp == 0) {
    r = lane < NW ? ws[lane] : T(0);
    r = warp_sum(r);
  }
  return r;
}

}  // namespace dphy
#endif
