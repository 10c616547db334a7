// Scoring of K sampled flows per image against the ground truth (evaluation.score_flows): per pixel, in one pass over the
// K samples, the mean flow, the spread of the samples around it and the end-point errors of the mean and of every sample;
// per image, the sums and counts the dataset-level metrics are built from (contract: include/flowdiff.h).
//
// Layout: block (c, b) owns the contiguous pixel chunk c of image b (kChunk pixels, so no block mixes images); a thread owns
// kPix pixels of it.  The loop runs over k outside and over the thread's pixels inside, so the per-sample EPE sum of
// sample k is one scalar per thread, reduced across the warp before k + 1: any K works with a fixed register budget.
// Every warp writes its (8 + K) float partials to the workspace; a second launch sums them per (image, column) in a fixed
// order in fp64.  No atomics: two launches on the same inputs give the same bits.
#include "fd_common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kPix = 8;                          // pixels per thread
constexpr int kChunk = kThreads * kPix;          // pixels per block
constexpr int kFixedCols = 8;
constexpr float kUnknownFlow = 1e9f;             // the .flo "unknown" marker; |gt| >= this (or NaN / inf) is invalid

struct EvalArgs {
  const float* samples;
  const float* gt;
  float* mean_out;
  float* spread_out;
  float* partials;
  float scale, gt_limit;
  int K;
  long HW;
};

// both components finite and below the "unknown" marker (NaN fails the comparison)
__device__ __forceinline__ bool valid_gt(float u, float v) { return fabsf(u) < kUnknownFlow && fabsf(v) < kUnknownFlow; }

template <int VEC>
__device__ __forceinline__ void load_vec(const float* p, float (&v)[VEC]) {
  if constexpr (VEC == 4) {
    const float4 q = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
  } else {
#pragma unroll
    for (int j = 0; j < VEC; ++j) v[j] = __ldg(p + j);
  }
}

template <int VEC>
__device__ __forceinline__ void store_vec(float* p, const float (&v)[VEC]) {
  if constexpr (VEC == 4) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
#pragma unroll
    for (int j = 0; j < VEC; ++j) p[j] = v[j];
  }
}

// VEC = 4: 16-byte loads and stores (HW % 4 == 0 and every pointer 16-byte aligned); VEC = 1 otherwise.
template <int VEC>
__global__ void __launch_bounds__(kThreads) flow_eval_kernel(EvalArgs a) {
  constexpr int kIter = kPix / VEC;
  const int b = blockIdx.y, K = a.K;
  const long HW = a.HW;
  const long p0 = (long)blockIdx.x * kChunk + threadIdx.x * VEC;   // pixel it * kThreads * VEC + j of this thread: p0 + ...
  const float* smp = a.samples + (long)b * K * 2 * HW;
  const bool has_gt = a.gt != nullptr;

  float gu[kIter][VEC], gv[kIter][VEC];
  float su[kIter][VEC], sv[kIter][VEC];              // running sums (the mean flow, summed in order k = 0 .. K-1)
  float mu[kIter][VEC], mv[kIter][VEC], m2[kIter][VEC];   // Welford mean and sum of squared deviations (the spread)
#pragma unroll
  for (int it = 0; it < kIter; ++it) {
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      gu[it][j] = gv[it][j] = 0.f;
      su[it][j] = sv[it][j] = mu[it][j] = mv[it][j] = m2[it][j] = 0.f;
    }
    if (p0 + it * kThreads * VEC < HW && has_gt) {
      load_vec<VEC>(a.gt + (long)b * 2 * HW + p0 + it * kThreads * VEC, gu[it]);
      load_vec<VEC>(a.gt + (long)b * 2 * HW + HW + p0 + it * kThreads * VEC, gv[it]);
    }
  }

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* part = a.partials + (((long)b * gridDim.x + blockIdx.x) * kWarps + warp) * (kFixedCols + K);
  for (int k = 0; k < K; ++k) {
    const float inv_n = 1.f / (float)(k + 1);
    const float* pu = smp + (long)k * 2 * HW;
    float epe_k = 0.f;
#pragma unroll
    for (int it = 0; it < kIter; ++it) {
      if (p0 + it * kThreads * VEC >= HW) continue;   // VEC = 4 implies HW % 4 == 0: a vector is wholly in or out
      float u[VEC], v[VEC];
      load_vec<VEC>(pu + p0 + it * kThreads * VEC, u);
      load_vec<VEC>(pu + HW + p0 + it * kThreads * VEC, v);
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        su[it][j] += u[j];
        sv[it][j] += v[j];
        const float du = u[j] - mu[it][j], dv = v[j] - mv[it][j];
        mu[it][j] = fmaf(du, inv_n, mu[it][j]);
        mv[it][j] = fmaf(dv, inv_n, mv[it][j]);
        m2[it][j] = fmaf(du, u[j] - mu[it][j], fmaf(dv, v[j] - mv[it][j], m2[it][j]));
        if (has_gt && valid_gt(gu[it][j], gv[it][j])) {                // a NaN sample at a valid pixel propagates into the sum
          const float eu = a.scale * u[j] - gu[it][j], ev = a.scale * v[j] - gv[it][j];
          epe_k += sqrtf(fmaf(eu, eu, ev * ev));
        }
      }
    }
    epe_k = fd_warp_sum(epe_k);
    if (lane == 0) part[kFixedCols + k] = epe_k;
  }

  // cols: 0 valid, 1 sum EPE(mean), 2-4 EPE < 1 / 3 / 5, 5 Fl outlier, 6 sum spread, 7 |gt| beyond gt_limit
  float acc[kFixedCols] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  const float inv_k = 1.f / (float)K;
#pragma unroll
  for (int it = 0; it < kIter; ++it) {
    if (p0 + it * kThreads * VEC >= HW) continue;   // VEC = 4 implies HW % 4 == 0: a vector is wholly in or out
    float fu[VEC], fv[VEC], sp[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      fu[j] = su[it][j] * inv_k * a.scale;
      fv[j] = sv[it][j] * inv_k * a.scale;
      sp[j] = a.scale * sqrtf(m2[it][j] * inv_k);
      if (has_gt && !valid_gt(gu[it][j], gv[it][j])) continue;
      acc[0] += 1.f;
      acc[6] += sp[j];
      if (has_gt) {
        const float eu = fu[j] - gu[it][j], ev = fv[j] - gv[it][j];
        const float epe = sqrtf(fmaf(eu, eu, ev * ev));
        const float mag = sqrtf(fmaf(gu[it][j], gu[it][j], gv[it][j] * gv[it][j]));
        acc[1] += epe;
        acc[2] += epe < 1.f ? 1.f : 0.f;
        acc[3] += epe < 3.f ? 1.f : 0.f;
        acc[4] += epe < 5.f ? 1.f : 0.f;
        acc[5] += (epe > 3.f && epe > 0.05f * mag) ? 1.f : 0.f;
        acc[7] += fmaxf(fabsf(gu[it][j]), fabsf(gv[it][j])) > a.gt_limit ? 1.f : 0.f;
      }
    }
    if (a.mean_out) {
      store_vec<VEC>(a.mean_out + (long)b * 2 * HW + p0 + it * kThreads * VEC, fu);
      store_vec<VEC>(a.mean_out + (long)b * 2 * HW + HW + p0 + it * kThreads * VEC, fv);
    }
    if (a.spread_out) store_vec<VEC>(a.spread_out + (long)b * HW + p0 + it * kThreads * VEC, sp);
  }
#pragma unroll
  for (int c = 0; c < kFixedCols; ++c) acc[c] = fd_warp_sum(acc[c]);
  if (lane == 0) {
#pragma unroll
    for (int c = 0; c < kFixedCols; ++c) part[c] = acc[c];
  }
}

// block (column, image): thread t sums the warp partials t, t + 256, ... in fp64, then a fixed tree over the threads
__global__ void __launch_bounds__(kThreads) flow_eval_finalize_kernel(const float* __restrict__ partials, int n_warps,
                                                                      int cols, double* __restrict__ per_image) {
  __shared__ double red[kThreads];
  const int c = blockIdx.x, b = blockIdx.y;
  const float* p = partials + (long)b * n_warps * cols + c;
  double s = 0.0;
  for (int i = threadIdx.x; i < n_warps; i += kThreads) s += (double)p[(long)i * cols];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = kThreads / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) per_image[(long)b * cols + c] = red[0];
}

long chunks_per_image(int H, int W) { return ((long)H * W + kChunk - 1) / kChunk; }

bool aligned16(const void* p) { return p == nullptr || (((uintptr_t)p) & 15) == 0; }

}  // namespace

extern "C" {

size_t fd_flow_eval_workspace_floats(int B, int K, int H, int W) {
  if (B <= 0 || K <= 0 || H <= 0 || W <= 0) return 0;
  return (size_t)B * (size_t)chunks_per_image(H, W) * kWarps * (size_t)(kFixedCols + K);
}

int fd_flow_eval(const float* samples, float scale, const float* gt, float gt_limit, float* mean_out, float* spread_out,
                 double* per_image, float* workspace, int B, int K, int H, int W, void* stream) {
  FD_REQUIRE(samples && per_image && workspace && B > 0 && K > 0 && H > 0 && W > 0, "flow_eval: bad argument");
  FD_REQUIRE(B <= 65535, "flow_eval: B = %d > 65535 images per launch", B);
  const long chunks = chunks_per_image(H, W);
  FD_REQUIRE(chunks * kWarps <= 0x7fffffffL && K <= 0x7fffffff - kFixedCols, "flow_eval: image or K too large");
  cudaStream_t st = (cudaStream_t)stream;
  EvalArgs a{samples, gt, mean_out, spread_out, workspace, scale, gt_limit, K, (long)H * W};
  const dim3 grid((unsigned)chunks, (unsigned)B);
  const bool v4 = (W % 4 == 0) && aligned16(samples) && aligned16(gt) && aligned16(mean_out) && aligned16(spread_out);
  if (v4)
    flow_eval_kernel<4><<<grid, kThreads, 0, st>>>(a);
  else
    flow_eval_kernel<1><<<grid, kThreads, 0, st>>>(a);
  FD_LAUNCH_CHECK();
  flow_eval_finalize_kernel<<<dim3(kFixedCols + K, B), kThreads, 0, st>>>(workspace, (int)(chunks * kWarps), kFixedCols + K,
                                                                         per_image);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

}  // extern "C"
