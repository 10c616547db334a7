// Shared helpers for libflowdiff.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/flowdiff.h"

#define FD_NUM_SMS 148

void fd_set_error(const char* fmt, ...);

#define FD_REQUIRE(cond, ...)                 \
  do {                                        \
    if (!(cond)) {                            \
      fd_set_error(__VA_ARGS__);              \
      return FD_EINVAL;                       \
    }                                         \
  } while (0)

#define FD_CUDA(call)                                                              \
  do {                                                                             \
    cudaError_t e__ = (call);                                                      \
    if (e__ != cudaSuccess) {                                                      \
      fd_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      return FD_ECUDA;                                                             \
    }                                                                              \
  } while (0)

extern unsigned long long g_fd_launches;   // kernels launched by this library (bench.py's gpu_launches)
#define FD_LAUNCH_CHECK()          \
  do {                             \
    ++g_fd_launches;               \
    FD_CUDA(cudaGetLastError());   \
  } while (0)

static inline int fd_ceil_div(long a, long b) { return (int)((a + b - 1) / b); }

// ---- diagnostic builds ----------------------------------------------------------------------------------------------
// A build with -DFD_DIAG (FD_DIAG=1 python -m opticalflowdiffusion_b200.build) compiles timing-isolation switches into the
// conv, LinearAttention, attention and warp-window kernels: a bit mask read once from FD_CONV_DBG, FD_LA_DBG, FD_ATTN_DBG or
// FD_WARP_WIN_DBG skips parts of the work (the results are garbage).  Every test of a mask is written `kDiag && (p.dbg & k)`,
// so the default build contains none of them.
#ifdef FD_DIAG
#include <stdlib.h>
constexpr bool kDiag = true;
static inline int fd_diag_bits(const char* name) {
  const char* e = getenv(name);
  return e ? atoi(e) : 0;
}
#else
constexpr bool kDiag = false;
static inline int fd_diag_bits(const char*) { return 0; }
#endif

__device__ __forceinline__ float fd_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float fd_warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// block-wide sum of up to NV values; result valid in thread 0. blockDim.x multiple of 32, <= 1024.
template <int NV>
__device__ __forceinline__ void fd_block_sum(float (&v)[NV], float* smem /* >= NV*32 floats */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = fd_warp_sum(v[i]);
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) smem[i * 32 + warp] = v[i];
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      float x = lane < nwarp ? smem[i * 32 + lane] : 0.f;
      v[i] = fd_warp_sum(x);
    }
  }
  __syncthreads();
}

__device__ __forceinline__ float fd_silu(float x) { return __fdividef(x, 1.f + __expf(-x)); }

__device__ __forceinline__ uint32_t fd_pack_bf16(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float2 fd_unpack_bf16(uint32_t u) {
  __nv_bfloat162 h = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(h);
}

// ---------------------------------------------------------------------------------------------
// scatter with in-thread and neighbour-lane merging.  Must be called by all 32 lanes of a warp.
// addr[k] < 0 marks "no contribution".  Entries are ordered left to right along the row, so equal
// addresses are adjacent whenever the flow is locally smooth.
// ---------------------------------------------------------------------------------------------
template <int N>
__device__ __forceinline__ void fd_scatter_merged(float* __restrict__ plane, const int (&addr)[N], const float (&val)[N]) {
  int haddr = -1, taddr = -1;
  float hval = 0.f, tval = 0.f;
  bool have_head = false;
#pragma unroll
  for (int k = 0; k < N; ++k) {
    if (addr[k] < 0) continue;
    if (addr[k] == taddr) {
      tval += val[k];
    } else {
      if (taddr >= 0) {
        if (!have_head) {
          haddr = taddr; hval = tval; have_head = true;
        } else {
          atomicAdd(plane + taddr, tval);
        }
      }
      taddr = addr[k];
      tval = val[k];
    }
  }
  if (!have_head) {  // zero or one group: it is the head, nothing is offered to the next lane
    haddr = taddr; hval = tval; taddr = -1; tval = 0.f;
  }
  const int lane = threadIdx.x & 31;
  // offer the tail group to lane+1; it absorbs it when its head hits the same address
  int raddr = __shfl_up_sync(0xffffffffu, taddr, 1);
  float rval = __shfl_up_sync(0xffffffffu, tval, 1);
  bool absorb = (lane > 0) && (raddr >= 0) && (raddr == haddr);
  if (absorb) hval += rval;
  const bool taken = __shfl_down_sync(0xffffffffu, (int)absorb, 1) != 0 && lane < 31;
  if (haddr >= 0) atomicAdd(plane + haddr, hval);
  if (taddr >= 0 && !taken) atomicAdd(plane + taddr, tval);
}

