// Micro-benchmark: the rate at which the L2 executes red.global.add (fp32) for the access pattern of the scatter kernels of
// BASELINE config #4 (forward splat, gradient of the sampled frame in the warp backward): one thread per source pixel of an
// 8 x 436 x 1024 batch, four bilinear taps around pixel + displacement.  It is the roofline denominator of those kernels: they
// move few bytes per pixel but issue 4 (pixel-interleaved, 128-bit) or 12-16 (planar, scalar) reductions per pixel.
//   pattern 0: displacement 0 (perfect locality)      pattern 1: white-noise displacement, |d| <= 12 px (config #4: sigma 4 px)
//   v4: one red.global.add.v4.f32 per tap into a (B, H, W, 4) buffer     s3: three scalar reductions per tap into 3 planes
// Build: nvcc -O3 -gencode arch=compute_100a,code=sm_100a -o red_rate red_rate.cu ; run: ./red_rate
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>

constexpr int B = 8, H = 436, W = 1024;

__device__ __forceinline__ uint32_t hash32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
  return x;
}

template <int NOISE, int VEC4>
__global__ void __launch_bounds__(256) red_kernel(float* __restrict__ buf, long npix) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += (long)gridDim.x * blockDim.x) {
    const int b = (int)(i / ((long)H * W));
    const int r = (int)(i - (long)b * H * W);
    int y = r / W, x = r - y * W;
    if (NOISE) {
      const uint32_t h = hash32((uint32_t)i);
      x += (int)(h % 25u) - 12;
      y += (int)((h >> 8) % 25u) - 12;
    }
    const float v = 1.0f;
    const bool okx0 = x >= 0 && x < W, okx1 = x + 1 >= 0 && x + 1 < W, oky0 = y >= 0 && y < H, oky1 = y + 1 >= 0 && y + 1 < H;
    if (VEC4) {
      float* cell = buf + (((long)b * H + y) * W + x) * 4;
      auto red4 = [&](float* dst) {
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(v), "f"(v), "f"(v), "f"(v) : "memory");
      };
      if (okx0 && oky0) red4(cell);
      if (okx1 && oky0) red4(cell + 4);
      if (okx0 && oky1) red4(cell + (long)W * 4);
      if (okx1 && oky1) red4(cell + (long)W * 4 + 4);
    } else {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        float* cell = buf + (((long)b * 3 + c) * H + y) * W + x;
        if (okx0 && oky0) atomicAdd(cell, v);
        if (okx1 && oky0) atomicAdd(cell + 1, v);
        if (okx0 && oky1) atomicAdd(cell + W, v);
        if (okx1 && oky1) atomicAdd(cell + W + 1, v);
      }
    }
  }
}

// Lane pairs share a pixel: lane 2j issues the west tap and lane 2j + 1 the east tap of the SAME row in ONE instruction, so the
// two 16-byte operands (adjacent cells) reach the L2 as one 32-byte sector operation whenever the cell column is even.
template <int NOISE>
__global__ void __launch_bounds__(256) red_pair_kernel(float* __restrict__ buf, long npix) {
  const int lane = threadIdx.x & 31, side = lane & 1;
  for (long i0 = (long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); i0 < npix; i0 += (long)gridDim.x * blockDim.x) {
    const long i = i0 + lane;
    int b = 0, x = -8, y = -8;
    if (i < npix) {
      b = (int)(i / ((long)H * W));
      const int r = (int)(i - (long)b * H * W);
      y = r / W;
      x = r - y * W;
      if (NOISE) {
        const uint32_t h = hash32((uint32_t)i);
        x += (int)(h % 25u) - 12;
        y += (int)((h >> 8) % 25u) - 12;
      }
    }
    const float v = 1.0f;
#pragma unroll
    for (int who = 0; who < 2; ++who) {                    // pixel of the even lane, then pixel of the odd lane
      const int src = (lane & ~1) | who;
      const int px = __shfl_sync(0xffffffffu, x, src), py = __shfl_sync(0xffffffffu, y, src), pb = __shfl_sync(0xffffffffu, b, src);
      const int cx = px + side;
      const bool okx = cx >= 0 && cx < W;
      float* cell = buf + (((long)pb * H + py) * W + cx) * 4;
      if (okx && py >= 0 && py < H)
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(cell), "f"(v), "f"(v), "f"(v), "f"(v) : "memory");
      if (okx && py + 1 >= 0 && py + 1 < H)
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(cell + (long)W * 4), "f"(v), "f"(v), "f"(v), "f"(v) : "memory");
    }
  }
}

template <int NOISE>
void run_pair(const char* name, float* buf, size_t bytes, int blocks_per_sm) {
  int sms = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  const long npix = (long)B * H * W;
  cudaEvent_t s, e;
  cudaEventCreate(&s);
  cudaEventCreate(&e);
  float best = 1e30f;
  for (int rep = 0; rep < 12; ++rep) {
    cudaMemsetAsync(buf, 0, bytes);
    cudaEventRecord(s);
    red_pair_kernel<NOISE><<<sms * blocks_per_sm, 256>>>(buf, npix);
    cudaEventRecord(e);
    cudaEventSynchronize(e);
    float ms;
    cudaEventElapsedTime(&ms, s, e);
    if (rep >= 2 && ms < best) best = ms;
  }
  const double reds = (double)npix * 4;
  printf("%-44s %2d blocks/SM: %8.1f us   %7.1f G reductions/s   %6.1f GB/s of reduction payload\n", name, blocks_per_sm,
         best * 1e3, reds / (best * 1e-3) * 1e-9, reds * 16 / (best * 1e-3) * 1e-9);
}

template <int NOISE, int VEC4>
void run(const char* name, float* buf, size_t bytes, int blocks_per_sm) {
  int sms = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  const long npix = (long)B * H * W;
  cudaEvent_t s, e;
  cudaEventCreate(&s);
  cudaEventCreate(&e);
  float best = 1e30f;
  for (int rep = 0; rep < 12; ++rep) {
    cudaMemsetAsync(buf, 0, bytes);
    cudaEventRecord(s);
    red_kernel<NOISE, VEC4><<<sms * blocks_per_sm, 256>>>(buf, npix);
    cudaEventRecord(e);
    cudaEventSynchronize(e);
    float ms;
    cudaEventElapsedTime(&ms, s, e);
    if (rep >= 2 && ms < best) best = ms;
  }
  const double reds = (double)npix * 4 * (VEC4 ? 1 : 3);
  printf("%-44s %2d blocks/SM: %8.1f us   %7.1f G reductions/s   %6.1f GB/s of reduction payload\n", name, blocks_per_sm,
         best * 1e3, reds / (best * 1e-3) * 1e-9, reds * (VEC4 ? 16 : 4) / (best * 1e-3) * 1e-9);
}

int main() {
  const size_t bytes = sizeof(float) * 4 * (size_t)B * H * W;
  float* buf;
  if (cudaMalloc(&buf, bytes) != cudaSuccess) { printf("alloc failed\n"); return 1; }
  printf("red.global.add rate, %d x %d x %d pixels, 4 taps per pixel (scripts/micro/red_rate.cu)\n", B, H, W);
  for (int bps : {8, 16}) {
    run<0, 1>("v4.f32, displacement 0", buf, bytes, bps);
    run<1, 1>("v4.f32, white-noise displacement +-12 px", buf, bytes, bps);
    run_pair<1>("v4.f32, white noise, lane pairs per row", buf, bytes, bps);
    run<0, 0>("3 x f32 planar, displacement 0", buf, bytes, bps);
    run<1, 0>("3 x f32 planar, white-noise +-12 px", buf, bytes, bps);
  }
  // the two bandwidth-bound passes that surround the scatter in fd_splat_fwd / fd_warp_bwd_win
  cudaEvent_t s, e;
  cudaEventCreate(&s);
  cudaEventCreate(&e);
  float best = 1e30f;
  for (int rep = 0; rep < 8; ++rep) {
    cudaEventRecord(s);
    cudaMemsetAsync(buf, 0, bytes);
    cudaEventRecord(e);
    cudaEventSynchronize(e);
    float ms;
    cudaEventElapsedTime(&ms, s, e);
    if (rep >= 2 && ms < best) best = ms;
  }
  printf("memset of the %.1f MB accumulation buffer: %.1f us\n", bytes * 1e-6, best * 1e3);
  cudaError_t err = cudaDeviceSynchronize();
  printf("status: %s\n", cudaGetErrorString(err));
  return err != cudaSuccess;
}
