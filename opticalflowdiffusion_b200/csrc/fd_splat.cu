// Forward splat ("softsplat") trio: softsplat_new.py:352-423 (out), :489-565 (ingrad),
// :600-700 (flowgrad) of the reference, plus warp_forward_flow's pre/post-processing
// (warp.py:121-156).  fp32 NCHW, flow channel 0 = dx, channel 1 = dy.
//
// B200 layout: the reference runs one thread per *element* and recomputes the geometry per
// channel; here one thread owns VEC (=4 when W % 4 == 0) consecutive pixels of a row, computes the
// remapped coordinate once and loops over channels, with 128-bit loads of flow / input.  The
// forward scatter merges equal target addresses inside a thread and with the neighbouring lane
// before issuing red.global.add.f32 (several source pixels land in one target cell whenever
// scale > 1 or the flow is smooth).
//
// The reference's scale/offset remap mixes float and double arithmetic and differs between the
// three kernels (SURVEY.md section 8a, rows S1-S3); every such quirk is kept:
//   out      : the ">= size-1" branch only when scale > 1                        (:374-390)
//   ingrad   : that branch always; X additionally applies "* offset_x"           (:515-532)
//   flowgrad : that branch always; Y uses "* offset_y" instead of the abs/% form; the derivative
//              factor is 1/scale only in the last branch ("freeze gradient") and channel 0 (d/dx)
//              is scaled by the Y factor, channel 1 by the X factor               (:626-672)
#include <initializer_list>

#include "fd_common.cuh"

namespace {

enum { KIND_OUT = 0, KIND_INGRAD = 1, KIND_FLOWGRAD = 2 };
enum { AXIS_X = 0, AXIS_Y = 1 };

template <int KIND, int AXIS>
__device__ __forceinline__ float splat_remap(float f, int size, int scale, int offset, float& dflt) {
  dflt = 0.f;
  const float fsize = (float)size;
  bool upper = (double)f >= (double)fsize - 1.0;
  if (KIND == KIND_OUT) upper = upper && (scale > 1);
  if (upper) {
    int k = abs(offset - (size % scale)) % scale;
    if (KIND == KIND_FLOWGRAD && AXIS == AXIS_Y) k = offset;
    float r = (float)((double)f + ((double)__fsub_rn(f, fsize) + 1.0) * (double)(float)k);
    if (KIND == KIND_INGRAD && AXIS == AXIS_X)
      r = (float)((double)r + ((double)__fsub_rn(r, fsize) + 1.0) * (double)(float)offset);
    return __fdiv_rn(__fsub_rn(r, (float)offset), (float)scale);
  }
  const float fo = __fsub_rn(f, (float)offset);
  if ((double)fo < 0.0) return fo;
  dflt = __fdiv_rn(1.0f, (float)scale);
  return __fdiv_rn(fo, (float)scale);
}

struct SplatTaps {
  float nw, ne, sw, se;
  float fx, fy;
  float dxx, dyy;
  int x0, y0;
  bool ok;                       // finite
  bool okx0, okx1, oky0, oky1;   // inside the target plane
};

template <int KIND>
__device__ __forceinline__ void splat_taps(float flow_x, float flow_y, int x, int y, int H, int W, int Ho, int Wo,
                                           int scale, int off_x, int off_y, SplatTaps& t) {
  float fx = __fadd_rn((float)x, flow_x);
  float fy = __fadd_rn((float)y, flow_y);
  t.ok = isfinite(fx) && isfinite(fy);
  if (!t.ok) { fx = 0.f; fy = 0.f; }
  fx = splat_remap<KIND, AXIS_X>(fx, W, scale, off_x, t.dxx);
  fy = splat_remap<KIND, AXIS_Y>(fy, H, scale, off_y, t.dyy);
  t.fx = fx;
  t.fy = fy;
  const float x0f = floorf(fx), y0f = floorf(fy);
  // the reference converts floor() to int; out-of-range values fail the bounds test either way
  const bool xr = x0f >= -2.f && x0f <= (float)Wo;
  const bool yr = y0f >= -2.f && y0f <= (float)Ho;
  t.x0 = xr ? (int)x0f : -4;
  t.y0 = yr ? (int)y0f : -4;
  const float x1 = (float)(t.x0 + 1), y1 = (float)(t.y0 + 1), x0 = (float)t.x0, y0 = (float)t.y0;
  t.nw = __fmul_rn(__fsub_rn(x1, fx), __fsub_rn(y1, fy));
  t.ne = __fmul_rn(__fsub_rn(fx, x0), __fsub_rn(y1, fy));
  t.sw = __fmul_rn(__fsub_rn(x1, fx), __fsub_rn(fy, y0));
  t.se = __fmul_rn(__fsub_rn(fx, x0), __fsub_rn(fy, y0));
  t.okx0 = t.ok && t.x0 >= 0 && t.x0 < Wo;
  t.okx1 = t.ok && t.x0 + 1 >= 0 && t.x0 + 1 < Wo;
  t.oky0 = t.y0 >= 0 && t.y0 < Ho;
  t.oky1 = t.y0 + 1 >= 0 && t.y0 + 1 < Ho;
}

template <int VEC>
struct SVec;
template <>
struct SVec<1> {
  float v[1];
  __device__ __forceinline__ void load(const float* p) { v[0] = __ldg(p); }
  __device__ __forceinline__ void store(float* p) const { *p = v[0]; }
};
template <>
struct SVec<4> {
  float v[4];
  __device__ __forceinline__ void load(const float* p) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  __device__ __forceinline__ void store(float* p) const {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};

template <int VEC>
__device__ __forceinline__ void s_item_to_byx(long item, int H, int W, int& b, int& y, int& x) {
  const int wq = W / VEC;
  x = (int)(item % wq) * VEC;
  const long r = item / wq;
  y = (int)(r % H);
  b = (int)(r / H);
}

template <int VEC>
__global__ void __launch_bounds__(256) splat_fwd_kernel(const float* __restrict__ in, const float* __restrict__ flow,
                                                        float* __restrict__ out, int B, int C, int H, int W, int Ho,
                                                        int Wo, int scale, int off_x, int off_y, long items) {
  const long HW = (long)H * W, HWo = (long)Ho * Wo;
  const int lane = threadIdx.x & 31;
  for (long base = (long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < items;
       base += (long)gridDim.x * blockDim.x) {
    const long item = base + lane;
    const bool valid = item < items;
    int b = 0, y = 0, x = 0;
    if (valid) s_item_to_byx<VEC>(item, H, W, b, y, x);
    const long pix = (long)y * W + x;
    SVec<VEC> fx, fy;
#pragma unroll
    for (int j = 0; j < VEC; ++j) fx.v[j] = fy.v[j] = 0.f;
    if (valid) {
      fx.load(flow + ((long)b * 2 + 0) * HW + pix);
      fy.load(flow + ((long)b * 2 + 1) * HW + pix);
    }
    SplatTaps t[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) splat_taps<KIND_OUT>(fx.v[j], fy.v[j], x + j, y, H, W, Ho, Wo, scale, off_x, off_y, t[j]);
    for (int c = 0; c < C; ++c) {
      SVec<VEC> a;
#pragma unroll
      for (int j = 0; j < VEC; ++j) a.v[j] = 0.f;
      if (valid) a.load(in + ((long)b * C + c) * HW + pix);
      int a0[2 * VEC], a1[2 * VEC];
      float v0[2 * VEC], v1[2 * VEC];
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const int r0 = t[j].y0 * Wo + t[j].x0;
        a0[2 * j] = (valid && t[j].okx0 && t[j].oky0) ? r0 : -1;
        a0[2 * j + 1] = (valid && t[j].okx1 && t[j].oky0) ? r0 + 1 : -1;
        a1[2 * j] = (valid && t[j].okx0 && t[j].oky1) ? r0 + Wo : -1;
        a1[2 * j + 1] = (valid && t[j].okx1 && t[j].oky1) ? r0 + Wo + 1 : -1;
        v0[2 * j] = __fmul_rn(a.v[j], t[j].nw);
        v0[2 * j + 1] = __fmul_rn(a.v[j], t[j].ne);
        v1[2 * j] = __fmul_rn(a.v[j], t[j].sw);
        v1[2 * j + 1] = __fmul_rn(a.v[j], t[j].se);
      }
      float* plane = out + ((long)b * C + c) * HWo;
      fd_scatter_merged<2 * VEC>(plane, a0, v0);
      fd_scatter_merged<2 * VEC>(plane, a1, v1);
    }
  }
}

__device__ __forceinline__ float tap_or_zero(const float* __restrict__ plane, bool ok, int idx) {
  return ok ? __ldg(plane + idx) : 0.f;
}

template <int VEC>
__global__ void __launch_bounds__(256) splat_ingrad_kernel(const float* __restrict__ flow,
                                                           const float* __restrict__ gout, float* __restrict__ gin,
                                                           int B, int C, int H, int W, int Ho, int Wo, int scale,
                                                           int off_x, int off_y, long items) {
  const long HW = (long)H * W, HWo = (long)Ho * Wo;
  for (long item = (long)blockIdx.x * blockDim.x + threadIdx.x; item < items; item += (long)gridDim.x * blockDim.x) {
    int b, y, x;
    s_item_to_byx<VEC>(item, H, W, b, y, x);
    const long pix = (long)y * W + x;
    SVec<VEC> fx, fy;
    fx.load(flow + ((long)b * 2 + 0) * HW + pix);
    fy.load(flow + ((long)b * 2 + 1) * HW + pix);
    SplatTaps t[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j)
      splat_taps<KIND_INGRAD>(fx.v[j], fy.v[j], x + j, y, H, W, Ho, Wo, scale, off_x, off_y, t[j]);
    for (int c = 0; c < C; ++c) {
      const float* plane = gout + ((long)b * C + c) * HWo;
      SVec<VEC> g;
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const int r0 = t[j].y0 * Wo + t[j].x0;
        float acc = 0.f;
        acc += tap_or_zero(plane, t[j].okx0 && t[j].oky0, r0) * t[j].nw;
        acc += tap_or_zero(plane, t[j].okx1 && t[j].oky0, r0 + 1) * t[j].ne;
        acc += tap_or_zero(plane, t[j].okx0 && t[j].oky1, r0 + Wo) * t[j].sw;
        acc += tap_or_zero(plane, t[j].okx1 && t[j].oky1, r0 + Wo + 1) * t[j].se;
        g.v[j] = acc;
      }
      g.store(gin + ((long)b * C + c) * HW + pix);
    }
  }
}

template <int VEC>
__global__ void __launch_bounds__(256) splat_flowgrad_kernel(const float* __restrict__ in,
                                                             const float* __restrict__ flow,
                                                             const float* __restrict__ gout,
                                                             float* __restrict__ gflow, int B, int C, int H, int W,
                                                             int Ho, int Wo, int scale, int off_x, int off_y,
                                                             long items) {
  const long HW = (long)H * W, HWo = (long)Ho * Wo;
  for (long item = (long)blockIdx.x * blockDim.x + threadIdx.x; item < items; item += (long)gridDim.x * blockDim.x) {
    int b, y, x;
    s_item_to_byx<VEC>(item, H, W, b, y, x);
    const long pix = (long)y * W + x;
    SVec<VEC> fx, fy;
    fx.load(flow + ((long)b * 2 + 0) * HW + pix);
    fy.load(flow + ((long)b * 2 + 1) * HW + pix);
    SplatTaps t[VEC];
    float gx[VEC], gy[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      splat_taps<KIND_FLOWGRAD>(fx.v[j], fy.v[j], x + j, y, H, W, Ho, Wo, scale, off_x, off_y, t[j]);
      gx[j] = gy[j] = 0.f;
    }
    for (int c = 0; c < C; ++c) {
      const float* plane = gout + ((long)b * C + c) * HWo;
      SVec<VEC> a;
      a.load(in + ((long)b * C + c) * HW + pix);
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const int r0 = t[j].y0 * Wo + t[j].x0;
        const float x0 = (float)t[j].x0, y0 = (float)t[j].y0, x1 = (float)(t[j].x0 + 1), y1 = (float)(t[j].y0 + 1);
        const float g_nw = tap_or_zero(plane, t[j].okx0 && t[j].oky0, r0);
        const float g_ne = tap_or_zero(plane, t[j].okx1 && t[j].oky0, r0 + 1);
        const float g_sw = tap_or_zero(plane, t[j].okx0 && t[j].oky1, r0 + Wo);
        const float g_se = tap_or_zero(plane, t[j].okx1 && t[j].oky1, r0 + Wo + 1);
        const float fxx = t[j].fx, fyy = t[j].fy;
        // channel 0 (d/dx): weights -(y1-fy), +(y1-fy), -(fy-y0), +(fy-y0), factor dfltYY (:664-668)
        gx[j] += g_nw * a.v[j] * (-1.f * (y1 - fyy)) * t[j].dyy;
        gx[j] += g_ne * a.v[j] * (+1.f * (y1 - fyy)) * t[j].dyy;
        gx[j] += g_sw * a.v[j] * (-1.f * (fyy - y0)) * t[j].dyy;
        gx[j] += g_se * a.v[j] * (+1.f * (fyy - y0)) * t[j].dyy;
        // channel 1 (d/dy): weights -(x1-fx), -(fx-x0), +(x1-fx), +(fx-x0), factor dfltXX (:670-675)
        gy[j] += g_nw * a.v[j] * ((x1 - fxx) * -1.f) * t[j].dxx;
        gy[j] += g_ne * a.v[j] * ((fxx - x0) * -1.f) * t[j].dxx;
        gy[j] += g_sw * a.v[j] * ((x1 - fxx) * +1.f) * t[j].dxx;
        gy[j] += g_se * a.v[j] * ((fxx - x0) * +1.f) * t[j].dxx;
      }
    }
    SVec<VEC> ox, oy;
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      ox.v[j] = t[j].ok ? gx[j] : 0.f;
      oy.v[j] = t[j].ok ? gy[j] : 0.f;
    }
    ox.store(gflow + ((long)b * 2 + 0) * HW + pix);
    oy.store(gflow + ((long)b * 2 + 1) * HW + pix);
  }
}

// ---------------------------------------------------------------------------------------------
// All scale^2 offsets of one pyramid level in ONE launch (FlowLearner's loss loops `for a in range(level): for b in
// range(level): softsplat(..., scale=level, offset=[a, b])`, flow_learner.py:184-196 -- 832 splat pairs per step).
// Offset index k = a * scale + b -> (off_x, off_y) = (a, b); outputs / output gradients are stacked pixel-interleaved, (K, B, Ho, Wo, 4).
// The per-offset arithmetic is the single-offset kernels' (same taps, same order); the two gather kernels sum the
// K contributions of a source pixel in registers instead of K separate passes.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) splat_fwd_multi_kernel(const float* __restrict__ in, const float* __restrict__ flow,
                                                              float* __restrict__ out, int B, int H, int W, int Ho,
                                                              int Wo, int scale, long items) {
  // Four input channels (r, g, b, weight); the stacked output is pixel-interleaved (K, B, Ho, Wo, 4), so a tap is one 128-bit
  // reduction.  The scatter is bound by the NUMBER of L2 reduction operations (at level L every output cell receives ~L^2
  // contributions per offset): per-channel scalar reductions made this kernel 64 % of a FlowLearner step (ncu launch list).
  // Measured and not kept: summing the lanes with equal footprints in registers first (match.any + 16 shuffles per group
  // member, leaders issue the reductions) cut the reductions ~10x at the high levels and made the objective SLOWER
  // (12.8 vs 9.6 ms): with vector reductions the kernel is bound by instruction issue, not by the L2 any more.
  const int k = blockIdx.y;
  const int off_x = k / scale, off_y = k - off_x * scale;
  const long HW = (long)H * W, HWo = (long)Ho * Wo;
  float* outk = out + (long)k * B * HWo * 4;
  for (long item = (long)blockIdx.x * blockDim.x + threadIdx.x; item < items; item += (long)gridDim.x * blockDim.x) {
    int b, y, x;
    s_item_to_byx<1>(item, H, W, b, y, x);
    const long pix = (long)y * W + x;
    const float fx = __ldg(flow + ((long)b * 2 + 0) * HW + pix), fy = __ldg(flow + ((long)b * 2 + 1) * HW + pix);
    SplatTaps t;
    splat_taps<KIND_OUT>(fx, fy, x, y, H, W, Ho, Wo, scale, off_x, off_y, t);
    float v[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) v[c] = __ldg(in + ((long)b * 4 + c) * HW + pix);
    float* cell = outk + (((long)b * Ho + t.y0) * Wo + t.x0) * 4;
    auto red4 = [&](float* dst, float wt) {
      asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(__fmul_rn(v[0], wt)), "f"(__fmul_rn(v[1], wt)),
                   "f"(__fmul_rn(v[2], wt)), "f"(__fmul_rn(v[3], wt))
                   : "memory");
    };
    if (t.okx0 && t.oky0) red4(cell, t.nw);
    if (t.okx1 && t.oky0) red4(cell + 4, t.ne);
    if (t.okx0 && t.oky1) red4(cell + (long)Wo * 4, t.sw);
    if (t.okx1 && t.oky1) red4(cell + (long)Wo * 4 + 4, t.se);
  }
}

template <int C>
__global__ void __launch_bounds__(256) splat_ingrad_multi_kernel(const float* __restrict__ flow, const float* __restrict__ gout,
                                                                 float* __restrict__ gin, int B, int H, int W, int Ho, int Wo,
                                                                 int scale, long items) {
  const long HW = (long)H * W, HWo = (long)Ho * Wo;
  const int K = scale * scale;
  for (long item = (long)blockIdx.x * blockDim.x + threadIdx.x; item < items; item += (long)gridDim.x * blockDim.x) {
    int b, y, x;
    s_item_to_byx<1>(item, H, W, b, y, x);
    const long pix = (long)y * W + x;
    const float fx = __ldg(flow + ((long)b * 2 + 0) * HW + pix), fy = __ldg(flow + ((long)b * 2 + 1) * HW + pix);
    float acc[C];
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = 0.f;
    for (int k = 0; k < K; ++k) {
      const int off_x = k / scale, off_y = k - off_x * scale;
      SplatTaps t;
      splat_taps<KIND_INGRAD>(fx, fy, x, y, H, W, Ho, Wo, scale, off_x, off_y, t);
      const int r0 = t.y0 * Wo + t.x0;
      const float4* gk = reinterpret_cast<const float4*>(gout) + ((long)k * B + b) * HWo;      // interleaved (K, B, Ho, Wo, 4)
      const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      const float4 g_nw = (t.okx0 && t.oky0) ? __ldg(gk + r0) : z, g_ne = (t.okx1 && t.oky0) ? __ldg(gk + r0 + 1) : z;
      const float4 g_sw = (t.okx0 && t.oky1) ? __ldg(gk + r0 + Wo) : z, g_se = (t.okx1 && t.oky1) ? __ldg(gk + r0 + Wo + 1) : z;
      const float gn[4][4] = {{g_nw.x, g_ne.x, g_sw.x, g_se.x}, {g_nw.y, g_ne.y, g_sw.y, g_se.y},
                              {g_nw.z, g_ne.z, g_sw.z, g_se.z}, {g_nw.w, g_ne.w, g_sw.w, g_se.w}};
#pragma unroll
      for (int c = 0; c < C; ++c) {
        float a = 0.f;
        a += gn[c][0] * t.nw;
        a += gn[c][1] * t.ne;
        a += gn[c][2] * t.sw;
        a += gn[c][3] * t.se;
        acc[c] += a;
      }
    }
#pragma unroll
    for (int c = 0; c < C; ++c) gin[((long)b * C + c) * HW + pix] = acc[c];
  }
}

template <int C>
__global__ void __launch_bounds__(256) splat_flowgrad_multi_kernel(const float* __restrict__ in, const float* __restrict__ flow,
                                                                   const float* __restrict__ gout, float* __restrict__ gflow,
                                                                   int B, int H, int W, int Ho, int Wo, int scale, long items) {
  const long HW = (long)H * W, HWo = (long)Ho * Wo;
  const int K = scale * scale;
  for (long item = (long)blockIdx.x * blockDim.x + threadIdx.x; item < items; item += (long)gridDim.x * blockDim.x) {
    int b, y, x;
    s_item_to_byx<1>(item, H, W, b, y, x);
    const long pix = (long)y * W + x;
    const float fx = __ldg(flow + ((long)b * 2 + 0) * HW + pix), fy = __ldg(flow + ((long)b * 2 + 1) * HW + pix);
    float a[C];
#pragma unroll
    for (int c = 0; c < C; ++c) a[c] = __ldg(in + ((long)b * C + c) * HW + pix);
    float gx = 0.f, gy = 0.f;
    bool ok = true;
    for (int k = 0; k < K; ++k) {
      const int off_x = k / scale, off_y = k - off_x * scale;
      SplatTaps t;
      splat_taps<KIND_FLOWGRAD>(fx, fy, x, y, H, W, Ho, Wo, scale, off_x, off_y, t);
      ok = t.ok;
      const int r0 = t.y0 * Wo + t.x0;
      const float x0 = (float)t.x0, y0 = (float)t.y0, x1 = (float)(t.x0 + 1), y1 = (float)(t.y0 + 1);
      const float4* gk = reinterpret_cast<const float4*>(gout) + ((long)k * B + b) * HWo;      // interleaved (K, B, Ho, Wo, 4)
      const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      const float4 q_nw = (t.okx0 && t.oky0) ? __ldg(gk + r0) : z, q_ne = (t.okx1 && t.oky0) ? __ldg(gk + r0 + 1) : z;
      const float4 q_sw = (t.okx0 && t.oky1) ? __ldg(gk + r0 + Wo) : z, q_se = (t.okx1 && t.oky1) ? __ldg(gk + r0 + Wo + 1) : z;
      const float gn[4][4] = {{q_nw.x, q_ne.x, q_sw.x, q_se.x}, {q_nw.y, q_ne.y, q_sw.y, q_se.y},
                              {q_nw.z, q_ne.z, q_sw.z, q_se.z}, {q_nw.w, q_ne.w, q_sw.w, q_se.w}};
      float kx = 0.f, ky = 0.f;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const float g_nw = gn[c][0], g_ne = gn[c][1], g_sw = gn[c][2], g_se = gn[c][3];
        kx += g_nw * a[c] * (-1.f * (y1 - t.fy)) * t.dyy;
        kx += g_ne * a[c] * (+1.f * (y1 - t.fy)) * t.dyy;
        kx += g_sw * a[c] * (-1.f * (t.fy - y0)) * t.dyy;
        kx += g_se * a[c] * (+1.f * (t.fy - y0)) * t.dyy;
        ky += g_nw * a[c] * ((x1 - t.fx) * -1.f) * t.dxx;
        ky += g_ne * a[c] * ((t.fx - x0) * -1.f) * t.dxx;
        ky += g_sw * a[c] * ((x1 - t.fx) * +1.f) * t.dxx;
        ky += g_se * a[c] * ((t.fx - x0) * +1.f) * t.dxx;
      }
      gx += kx;
      gy += ky;
    }
    gflow[((long)b * 2 + 0) * HW + pix] = ok ? gx : 0.f;
    gflow[((long)b * 2 + 1) * HW + pix] = ok ? gy : 0.f;
  }
}

// warp_forward_flow pre-processing (warp.py:122-126, softsplat_new.py:301-302):
// ten_in[:, :C] = nan_to_zero(first) * w ; ten_in[:, C] = w ; w = any_c(isnan(first)) ? 0 : 1
__global__ void __launch_bounds__(256) splat_prepare_kernel(const float* __restrict__ first, float* __restrict__ ten_in,
                                                            int B, int C, long HW) {
  const long total = (long)B * HW;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long b = i / HW, p = i % HW;
    bool any_nan = false;
    for (int c = 0; c < C; ++c) any_nan |= isnan(__ldg(first + (b * C + c) * HW + p));
    const float w = any_nan ? 0.f : 1.f;
    for (int c = 0; c < C; ++c) {
      float v = __ldg(first + (b * C + c) * HW + p);
      if (isnan(v)) v = 0.f;
      ten_in[(b * (C + 1) + c) * HW + p] = v * w;
    }
    ten_in[(b * (C + 1) + C) * HW + p] = w;
  }
}

// warp_forward_flow post-processing (warp.py:139-156): img = wsum > 0 ? splat[:, :C] : NaN
__global__ void __launch_bounds__(256) splat_finish_kernel(const float* __restrict__ splat, float* __restrict__ img,
                                                           int B, int C, long HW, int set_nans) {
  const long total = (long)B * HW;
  const float qnan = __int_as_float(0x7fc00000);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long b = i / HW, p = i % HW;
    const float w = __ldg(splat + (b * (C + 1) + C) * HW + p);
    for (int c = 0; c < C; ++c) {
      const float v = __ldg(splat + (b * (C + 1) + c) * HW + p);
      img[(b * C + c) * HW + p] = (!set_nans || w > 0.f) ? v : qnan;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// warp_forward_flow for three-channel images as TWO launches (prepare + splat + finish of the generic path fused):
//   * the accumulation buffer is pixel-interleaved (B, Ho, Wo, 4) = (r, g, b, weight), so a tap is ONE 128-bit
//     red.global.add.v4.f32 instead of four scalar reductions on four planes -- the scatter of the config-#4 flow is bound by
//     the number of L2 reduction operations (57 M scalar ones per call at 8 x 436 x 1024), not by bytes;
//   * NaN -> weight 0 and the weight channel (splat_prepare) are computed on the fly; ten_in is written only when the caller
//     keeps it for the backward; NaN source pixels (all four values zero) issue no reductions at all;
//   * the finish pass reads the interleaved sums once and writes the planar image (holes -> NaN) and the weight-sum plane.
// Same tap geometry and products as splat_fwd_kernel (splat_taps, __fmul_rn); the sums differ by the order of the atomics only.
// ---------------------------------------------------------------------------------------------
template <bool WRITE_IN>
__global__ void __launch_bounds__(256) splat_fwd3_kernel(const float* __restrict__ first, const float* __restrict__ flow,
                                                         float* __restrict__ ten_in, float* __restrict__ acc, int B, int H, int W,
                                                         int Ho, int Wo, int scale, int off_x, int off_y, unsigned segs,
                                                         unsigned jobs) {
  const long HW = (long)H * W;
  for (unsigned job = blockIdx.x; job < jobs; job += gridDim.x) {
    const unsigned row = job / segs, seg = job - row * segs;
    const unsigned b = row / (unsigned)H;
    const int y = (int)(row - b * (unsigned)H), x = (int)(seg * blockDim.x + threadIdx.x);
    if (x >= W) continue;
    const int pix = y * W + x;
    const float fx = __ldg(flow + ((long)b * 2 + 0) * HW + pix), fy = __ldg(flow + ((long)b * 2 + 1) * HW + pix);
    float v[3];
    bool any_nan = false;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      v[c] = __ldg(first + ((long)b * 3 + c) * HW + pix);
      any_nan |= isnan(v[c]);
    }
    const float w = any_nan ? 0.f : 1.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) v[c] = isnan(v[c]) ? 0.f : v[c] * w;
    if (WRITE_IN) {
#pragma unroll
      for (int c = 0; c < 3; ++c) ten_in[((long)b * 4 + c) * HW + pix] = v[c];
      ten_in[((long)b * 4 + 3) * HW + pix] = w;
    }
    if (any_nan) continue;                         // four zeros: nothing to add
    SplatTaps t;
    splat_taps<KIND_OUT>(fx, fy, x, y, H, W, Ho, Wo, scale, off_x, off_y, t);
    float* cell = acc + (((long)b * Ho + t.y0) * Wo + t.x0) * 4;
    auto red4 = [&](float* dst, float wt) {
      asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(__fmul_rn(v[0], wt)), "f"(__fmul_rn(v[1], wt)),
                   "f"(__fmul_rn(v[2], wt)), "f"(__fmul_rn(w, wt))
                   : "memory");
    };
    if (t.okx0 && t.oky0) red4(cell, t.nw);
    if (t.okx1 && t.oky0) red4(cell + 4, t.ne);
    if (t.okx0 && t.oky1) red4(cell + (long)Wo * 4, t.sw);
    if (t.okx1 && t.oky1) red4(cell + (long)Wo * 4 + 4, t.se);
  }
}

__global__ void __launch_bounds__(256) splat_finish3_kernel(const float* __restrict__ acc, float* __restrict__ img,
                                                            float* __restrict__ wsum, int B, long HWo, int set_nans) {
  const long total = (long)B * HWo;
  const float qnan = __int_as_float(0x7fc00000);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long b = i / HWo, p = i - b * HWo;
    const float4 a = __ldg(reinterpret_cast<const float4*>(acc) + i);
    const bool keep = !set_nans || a.w > 0.f;
    img[(b * 3 + 0) * HWo + p] = keep ? a.x : qnan;
    img[(b * 3 + 1) * HWo + p] = keep ? a.y : qnan;
    img[(b * 3 + 2) * HWo + p] = keep ? a.z : qnan;
    if (wsum != nullptr) wsum[i] = a.w;
  }
}

// fd_splat_fwd for 3 or 4 input channels through the same pixel-interleaved accumulation (one 128-bit reduction per tap; a
// fourth channel of zeros for C = 3), then a planar copy-out.  Same products as splat_fwd_kernel (which every other channel
// count runs); the sums differ by the order of the atomics only.
template <int C>
__global__ void __launch_bounds__(256) splat_fwd_il_kernel(const float* __restrict__ in, const float* __restrict__ flow,
                                                           float* __restrict__ acc, int B, int H, int W, int Ho, int Wo, int scale,
                                                           int off_x, int off_y, unsigned segs, unsigned jobs) {
  const long HW = (long)H * W;
  for (unsigned job = blockIdx.x; job < jobs; job += gridDim.x) {
    const unsigned row = job / segs, seg = job - row * segs;
    const unsigned b = row / (unsigned)H;
    const int y = (int)(row - b * (unsigned)H), x = (int)(seg * blockDim.x + threadIdx.x);
    if (x >= W) continue;
    const int pix = y * W + x;
    const float fx = __ldg(flow + ((long)b * 2 + 0) * HW + pix), fy = __ldg(flow + ((long)b * 2 + 1) * HW + pix);
    float v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int c = 0; c < C; ++c) v[c] = __ldg(in + ((long)b * C + c) * HW + pix);
    SplatTaps t;
    splat_taps<KIND_OUT>(fx, fy, x, y, H, W, Ho, Wo, scale, off_x, off_y, t);
    float* cell = acc + (((long)b * Ho + t.y0) * Wo + t.x0) * 4;
    auto red4 = [&](float* dst, float wt) {
      asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(__fmul_rn(v[0], wt)), "f"(__fmul_rn(v[1], wt)),
                   "f"(__fmul_rn(v[2], wt)), "f"(C == 4 ? __fmul_rn(v[3], wt) : 0.f)
                   : "memory");
    };
    if (t.okx0 && t.oky0) red4(cell, t.nw);
    if (t.okx1 && t.oky0) red4(cell + 4, t.ne);
    if (t.okx0 && t.oky1) red4(cell + (long)Wo * 4, t.sw);
    if (t.okx1 && t.oky1) red4(cell + (long)Wo * 4 + 4, t.se);
  }
}

template <int C>
__global__ void __launch_bounds__(256) il_to_planes_kernel(const float* __restrict__ acc, float* __restrict__ out, int B, long HWo) {
  const long total = (long)B * HWo;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long b = i / HWo, p = i - b * HWo;
    const float4 a = __ldg(reinterpret_cast<const float4*>(acc) + i);
    out[(b * C + 0) * HWo + p] = a.x;
    out[(b * C + 1) * HWo + p] = a.y;
    out[(b * C + 2) * HWo + p] = a.z;
    if (C == 4) out[(b * C + 3) * HWo + p] = a.w;
  }
}

// 128-bit accesses need 16-byte aligned planes (a view at an odd float offset is a legal argument)
bool al16(std::initializer_list<const void*> ptrs) {
  for (const void* q : ptrs)
    if (q != nullptr && (reinterpret_cast<uintptr_t>(q) & 15) != 0) return false;
  return true;
}

int sgrid(long items) {
  long blocks = (items + 255) / 256;
  const long cap = (long)FD_NUM_SMS * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

int check(int B, int C, int H, int W, int scale, int off_x, int off_y) {
  FD_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "splat: non-positive dimension");
  FD_REQUIRE(scale >= 1 && H / scale > 0 && W / scale > 0, "splat: bad scale %d for %dx%d", scale, H, W);
  FD_REQUIRE(off_x >= 0 && off_y >= 0, "splat: offsets must be reduced modulo scale (warp.py:129)");
  FD_REQUIRE((long)H * W < (1L << 31), "splat: plane too large");
  return FD_OK;
}

}  // namespace

extern "C" {

size_t fd_splat_fwd_workspace_floats(int B, int C, int H, int W, int scale) {
  return (C == 3 || C == 4) ? (size_t)4 * B * (H / scale) * (W / scale) : 0;
}

int fd_splat_fwd(const float* in, const float* flow, float* out, float* workspace, int B, int C, int H, int W, int scale,
                 int off_x, int off_y, void* stream) {
  if (int e = check(B, C, H, W, scale, off_x, off_y)) return e;
  FD_REQUIRE(in && flow && out, "splat_fwd: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int Ho = H / scale, Wo = W / scale;
  if (C != 3 && C != 4) {
    FD_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)B * C * Ho * Wo, st));
    if (W % 4 == 0 && al16({in, flow})) {
      const long items = (long)B * H * (W / 4);
      splat_fwd_kernel<4><<<sgrid(items), 256, 0, st>>>(in, flow, out, B, C, H, W, Ho, Wo, scale, off_x, off_y, items);
    } else {
      const long items = (long)B * H * W;
      splat_fwd_kernel<1><<<sgrid(items), 256, 0, st>>>(in, flow, out, B, C, H, W, Ho, Wo, scale, off_x, off_y, items);
    }
    FD_LAUNCH_CHECK();
    return FD_OK;
  }
  FD_REQUIRE(workspace != nullptr && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0,
             "splat_fwd: C = %d needs a 16-byte aligned workspace of fd_splat_fwd_workspace_floats floats", C);
  FD_CUDA(cudaMemsetAsync(workspace, 0, sizeof(float) * 4 * (size_t)B * Ho * Wo, st));
  const unsigned segs = (unsigned)((W + 255) / 256);
  const long jobs = (long)B * H * segs;
  FD_REQUIRE(jobs < (1L << 31), "splat_fwd: too many row segments");
  long grid = jobs;
  if (grid > (long)FD_NUM_SMS * 16) grid = (long)FD_NUM_SMS * 16;
  if (C == 3) {
    splat_fwd_il_kernel<3><<<(unsigned)grid, 256, 0, st>>>(in, flow, workspace, B, H, W, Ho, Wo, scale, off_x, off_y, segs, (unsigned)jobs);
    FD_LAUNCH_CHECK();
    il_to_planes_kernel<3><<<sgrid((long)B * Ho * Wo), 256, 0, st>>>(workspace, out, B, (long)Ho * Wo);
  } else {
    splat_fwd_il_kernel<4><<<(unsigned)grid, 256, 0, st>>>(in, flow, workspace, B, H, W, Ho, Wo, scale, off_x, off_y, segs, (unsigned)jobs);
    FD_LAUNCH_CHECK();
    il_to_planes_kernel<4><<<sgrid((long)B * Ho * Wo), 256, 0, st>>>(workspace, out, B, (long)Ho * Wo);
  }
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_forward_warp_sum3(const float* first, const float* flow, float* ten_in, float* acc, float* img, float* wsum, int B, int H,
                         int W, int scale, int off_x, int off_y, int set_nans, void* stream) {
  if (int e = check(B, 3, H, W, scale, off_x, off_y)) return e;
  FD_REQUIRE(first && flow && acc && img, "forward_warp_sum3: null pointer");
  FD_REQUIRE((reinterpret_cast<uintptr_t>(acc) & 15) == 0, "forward_warp_sum3: the accumulation buffer must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int Ho = H / scale, Wo = W / scale;
  FD_CUDA(cudaMemsetAsync(acc, 0, sizeof(float) * 4 * (size_t)B * Ho * Wo, st));
  const unsigned segs = (unsigned)((W + 255) / 256);
  const long jobs = (long)B * H * segs;
  FD_REQUIRE(jobs < (1L << 31), "forward_warp_sum3: too many row segments");
  long grid = jobs;
  if (grid > (long)FD_NUM_SMS * 16) grid = (long)FD_NUM_SMS * 16;
  if (ten_in != nullptr)
    splat_fwd3_kernel<true><<<(unsigned)grid, 256, 0, st>>>(first, flow, ten_in, acc, B, H, W, Ho, Wo, scale, off_x, off_y, segs,
                                                             (unsigned)jobs);
  else
    splat_fwd3_kernel<false><<<(unsigned)grid, 256, 0, st>>>(first, flow, nullptr, acc, B, H, W, Ho, Wo, scale, off_x, off_y, segs,
                                                              (unsigned)jobs);
  FD_LAUNCH_CHECK();
  splat_finish3_kernel<<<sgrid((long)B * Ho * Wo), 256, 0, st>>>(acc, img, wsum, B, (long)Ho * Wo, set_nans);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_splat_ingrad(const float* flow, const float* gout, float* gin, int B, int C, int H, int W, int scale,
                    int off_x, int off_y, void* stream) {
  if (int e = check(B, C, H, W, scale, off_x, off_y)) return e;
  FD_REQUIRE(flow && gout && gin, "splat_ingrad: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int Ho = H / scale, Wo = W / scale;
  if (W % 4 == 0 && al16({flow, gin})) {
    const long items = (long)B * H * (W / 4);
    splat_ingrad_kernel<4><<<sgrid(items), 256, 0, st>>>(flow, gout, gin, B, C, H, W, Ho, Wo, scale, off_x, off_y, items);
  } else {
    const long items = (long)B * H * W;
    splat_ingrad_kernel<1><<<sgrid(items), 256, 0, st>>>(flow, gout, gin, B, C, H, W, Ho, Wo, scale, off_x, off_y, items);
  }
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_splat_flowgrad(const float* in, const float* flow, const float* gout, float* gflow, int B, int C, int H, int W,
                      int scale, int off_x, int off_y, void* stream) {
  if (int e = check(B, C, H, W, scale, off_x, off_y)) return e;
  FD_REQUIRE(in && flow && gout && gflow, "splat_flowgrad: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int Ho = H / scale, Wo = W / scale;
  if (W % 4 == 0 && al16({in, flow, gflow})) {
    const long items = (long)B * H * (W / 4);
    splat_flowgrad_kernel<4><<<sgrid(items), 256, 0, st>>>(in, flow, gout, gflow, B, C, H, W, Ho, Wo, scale, off_x, off_y, items);
  } else {
    const long items = (long)B * H * W;
    splat_flowgrad_kernel<1><<<sgrid(items), 256, 0, st>>>(in, flow, gout, gflow, B, C, H, W, Ho, Wo, scale, off_x, off_y, items);
  }
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_splat_fwd_multi(const float* in, const float* flow, float* out, int B, int C, int H, int W, int scale, void* stream) {
  if (int e = check(B, C, H, W, scale, 0, 0)) return e;
  FD_REQUIRE(in && flow && out && scale * scale <= 65535, "splat_fwd_multi: bad argument");
  FD_REQUIRE(C == 4, "splat_fwd_multi: built for the 4-channel soft splat input (3 colours + weight), got C=%d", C);
  FD_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "splat_fwd_multi: out must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int Ho = H / scale, Wo = W / scale, K = scale * scale;
  FD_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)K * B * C * Ho * Wo, st));
  const long items = (long)B * H * W;
  int gx = sgrid(items);
  const int cap = (FD_NUM_SMS * 16 + K - 1) / K;
  if (gx > cap) gx = cap;
  splat_fwd_multi_kernel<<<dim3(gx, K), 256, 0, st>>>(in, flow, out, B, H, W, Ho, Wo, scale, items);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_splat_ingrad_multi(const float* flow, const float* gout, float* gin, int B, int C, int H, int W, int scale,
                          void* stream) {
  if (int e = check(B, C, H, W, scale, 0, 0)) return e;
  FD_REQUIRE(flow && gout && gin, "splat_ingrad_multi: null pointer");
  FD_REQUIRE(C == 4, "splat_ingrad_multi: built for the 4-channel soft splat input (3 colours + weight), got C=%d", C);
  FD_REQUIRE((reinterpret_cast<uintptr_t>(gout) & 15) == 0, "splat_ingrad_multi: gout must be 16-byte aligned");
  const long items = (long)B * H * W;
  splat_ingrad_multi_kernel<4><<<sgrid(items), 256, 0, (cudaStream_t)stream>>>(flow, gout, gin, B, H, W, H / scale, W / scale,
                                                                             scale, items);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_splat_flowgrad_multi(const float* in, const float* flow, const float* gout, float* gflow, int B, int C, int H, int W,
                            int scale, void* stream) {
  if (int e = check(B, C, H, W, scale, 0, 0)) return e;
  FD_REQUIRE(in && flow && gout && gflow, "splat_flowgrad_multi: null pointer");
  FD_REQUIRE(C == 4, "splat_flowgrad_multi: built for the 4-channel soft splat input (3 colours + weight), got C=%d", C);
  const long items = (long)B * H * W;
  splat_flowgrad_multi_kernel<4><<<sgrid(items), 256, 0, (cudaStream_t)stream>>>(in, flow, gout, gflow, B, H, W, H / scale,
                                                                               W / scale, scale, items);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_splat_prepare(const float* first, float* ten_in, int B, int C, int HW, void* stream) {
  FD_REQUIRE(first && ten_in && B > 0 && C > 0 && HW > 0, "splat_prepare: bad argument");
  splat_prepare_kernel<<<sgrid((long)B * HW), 256, 0, (cudaStream_t)stream>>>(first, ten_in, B, C, HW);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_splat_finish(const float* splat, float* img, int B, int C, int HW, int set_nans, void* stream) {
  FD_REQUIRE(splat && img && B > 0 && C > 0 && HW > 0, "splat_finish: bad argument");
  splat_finish_kernel<<<sgrid((long)B * HW), 256, 0, (cudaStream_t)stream>>>(splat, img, B, C, HW, set_nans);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

}  // extern "C"
