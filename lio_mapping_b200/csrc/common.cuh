// lio_mapping_b200 — shared device/host helpers for the sm_100a kernels behind the C-ABI.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include "../../include/lio_b200.h"

#define LIO_CUDA_OK(expr)                                                                   \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess) {                                                                \
      lio_set_last_error(__FILE__, __LINE__, cudaGetErrorString(_e));                       \
      return LIO_ERR_CUDA;                                                                  \
    }                                                                                       \
  } while (0)

void lio_set_last_error(const char *file, int line, const char *msg);

namespace lio {

constexpr int kWarp = 32;

// What one process call cost the host (lio_po_last_stats / lio_pm_last_stats): kernel launches, stream synchronisations
// and the bytes of every host<->device copy the call enqueued.
struct CallStats {
  long long launches = 0, syncs = 0, h2d = 0, d2h = 0;
  void reset() { launches = syncs = h2d = d2h = 0; }
};
inline cudaError_t stats_h2d(CallStats &s, void *dst, const void *src, size_t bytes, cudaStream_t st) {
  s.h2d += (long long)bytes;
  return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st);
}
inline cudaError_t stats_d2h(CallStats &s, void *dst, const void *src, size_t bytes, cudaStream_t st) {
  s.d2h += (long long)bytes;
  return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st);
}
inline cudaError_t stats_sync(CallStats &s, cudaStream_t st) {
  ++s.syncs;
  return cudaStreamSynchronize(st);
}

__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ unsigned warp_id() { return threadIdx.x >> 5; }

// Inclusive warp scan (int).
__device__ __forceinline__ int warp_scan_incl(int v) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, v, o);
    if ((int)lane_id() >= o) v += t;
  }
  return v;
}

// Block-wide exclusive scan for blockDim.x <= 1024; `smem` needs 33 ints.  Returns the exclusive
// prefix of v; *total receives the block sum.  All threads must call.
__device__ __forceinline__ int block_scan_excl(int v, int *smem, int *total) {
  int incl = warp_scan_incl(v);
  if (lane_id() == 31) smem[warp_id()] = incl;
  __syncthreads();
  if (warp_id() == 0) {
    int nw = (blockDim.x + 31) >> 5;
    int w = (int)lane_id() < nw ? smem[lane_id()] : 0;
    int wi = warp_scan_incl(w);
    smem[lane_id()] = wi - w;
    if ((int)lane_id() == nw - 1) smem[32] = wi;
  }
  __syncthreads();
  int r = smem[warp_id()] + incl - v;
  *total = smem[32];
  __syncthreads();
  return r;
}

__device__ __forceinline__ float4 ld_f4(const float4 *p) { return __ldg(p); }

}  // namespace lio
