// Diffusion scheduler updates and the NaN-aware MSE loss.
//   q_sample          denoising_diffusion.py:806-812
//   DDIM update       denoising_diffusion.py:653-656 (clamp), 595-599 (eps from x0), 757-767
//   DDPM update       denoising_diffusion.py:666-698, 613-623
//   DPM-Solver++      multistep data-prediction update, orders 1-3 (Lu et al., arXiv:2211.01095); not in the reference
//   nan_mse/nanmean   warp.py:260-271, denoising_diffusion.py:906-908,973
// Pure streaming kernels (HBM roofline): 128-bit accesses, one pass, every per-step scalar is a
// kernel argument computed on the host from the fp32 schedule tables, so the whole update is one
// launch instead of the reference's ~12 ATen kernels.  The arithmetic uses explicit
// round-to-nearest mul/add (no FMA contraction) in the reference's operation order, which keeps
// the update bit-identical to the fp32 PyTorch result given the same model output.
#include "fd_common.cuh"

namespace {

int egrid(long items) {
  long blocks = (items + 255) / 256;
  const long cap = (long)FD_NUM_SMS * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

__device__ __forceinline__ float clamp1(float v) {
  // torch.clamp(min=-1, max=1): min(max(v, -1), 1); NaN propagates
  if (v != v) return v;
  return fminf(fmaxf(v, -1.f), 1.f);
}

__global__ void __launch_bounds__(256) q_sample_kernel(const float* __restrict__ x0, const float* __restrict__ noise,
                                                       const int64_t* __restrict__ t, const float* __restrict__ sqrt_ac,
                                                       const float* __restrict__ sqrt_1mac, float* __restrict__ out,
                                                       int B, long per_sample) {
  const long total = (long)B * per_sample;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int b = (int)(i / per_sample);
    const long tb = t[b];
    const float a = __ldg(sqrt_ac + tb), s = __ldg(sqrt_1mac + tb);
    out[i] = __fadd_rn(__fmul_rn(a, __ldg(x0 + i)), __fmul_rn(s, __ldg(noise + i)));
  }
}

struct DdimArgs {
  float recip, recipm1, sqrt_alpha_next, c, sigma;
  int last;
};

__device__ __forceinline__ float ddim_one(float x, float mo, float nz, bool has_noise, const DdimArgs& a, float& x0o) {
  const float x0 = clamp1(mo);
  x0o = x0;
  if (a.last) return x0;
  const float eps = __fdiv_rn(__fsub_rn(__fmul_rn(a.recip, x), x0), a.recipm1);
  float r = __fadd_rn(__fmul_rn(x0, a.sqrt_alpha_next), __fmul_rn(a.c, eps));
  if (has_noise) r = __fadd_rn(r, __fmul_rn(a.sigma, nz));
  return r;
}

template <int VEC>
__global__ void __launch_bounds__(256) ddim_kernel(const float* __restrict__ x, const float* __restrict__ mo,
                                                   const float* __restrict__ noise, float* __restrict__ xn,
                                                   float* __restrict__ x0_out, long n, DdimArgs a) {
  const long items = n / VEC;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < items; i += (long)gridDim.x * blockDim.x) {
    if (VEC == 4) {
      const float4 xv = reinterpret_cast<const float4*>(x)[i];
      const float4 mv = __ldg(reinterpret_cast<const float4*>(mo) + i);
      float4 nv = make_float4(0.f, 0.f, 0.f, 0.f);
      if (noise) nv = __ldg(reinterpret_cast<const float4*>(noise) + i);
      float4 r, z;
      r.x = ddim_one(xv.x, mv.x, nv.x, noise != nullptr, a, z.x);
      r.y = ddim_one(xv.y, mv.y, nv.y, noise != nullptr, a, z.y);
      r.z = ddim_one(xv.z, mv.z, nv.z, noise != nullptr, a, z.z);
      r.w = ddim_one(xv.w, mv.w, nv.w, noise != nullptr, a, z.w);
      reinterpret_cast<float4*>(xn)[i] = r;
      if (x0_out) reinterpret_cast<float4*>(x0_out)[i] = z;
    } else {
      float z;
      const float r = ddim_one(x[i], __ldg(mo + i), noise ? __ldg(noise + i) : 0.f, noise != nullptr, a, z);
      xn[i] = r;
      if (x0_out) x0_out[i] = z;
    }
  }
}

// DPM-Solver++ multistep (data prediction, deterministic): x_next = cx*x + c0*D0 + c1*D1 + c2*D2 with D0 = clamp(mo).
// A term whose coefficient is 0 is not evaluated, so a NaN in an unused history slot cannot leak in as 0*NaN.
struct DpmppArgs {
  float cx, c0, c1, c2;
  int last;
};

__device__ __forceinline__ float dpmpp_one(float x, float mo, float d1, float d2, const DpmppArgs& a, float& d0o) {
  const float d0 = clamp1(mo);
  d0o = d0;
  if (a.last) return d0;
  float r = __fadd_rn(__fmul_rn(a.cx, x), __fmul_rn(a.c0, d0));
  if (a.c1 != 0.f) r = __fadd_rn(r, __fmul_rn(a.c1, d1));
  if (a.c2 != 0.f) r = __fadd_rn(r, __fmul_rn(a.c2, d2));
  return r;
}

// x / x_next and d_hist2 / d_out may alias (each element is read, then written, by the same thread): no __restrict__
// and no read-only-cache loads on those four.
template <int VEC>
__global__ void __launch_bounds__(256) dpmpp_kernel(const float* x, const float* __restrict__ mo,
                                                    const float* __restrict__ d1, const float* d2, float* xn,
                                                    float* d_out, long n, DpmppArgs a) {
  const long items = n / VEC;
  const long stride = (long)gridDim.x * blockDim.x;
  const long tid = (long)blockIdx.x * blockDim.x + threadIdx.x;
  for (long i = tid; i < items; i += stride) {
    if (VEC == 4) {
      const float4 xv = reinterpret_cast<const float4*>(x)[i];
      const float4 mv = __ldg(reinterpret_cast<const float4*>(mo) + i);
      float4 h1 = make_float4(0.f, 0.f, 0.f, 0.f), h2 = h1;
      if (d1) h1 = __ldg(reinterpret_cast<const float4*>(d1) + i);
      if (d2) h2 = reinterpret_cast<const float4*>(d2)[i];
      float4 r, z;
      r.x = dpmpp_one(xv.x, mv.x, h1.x, h2.x, a, z.x);
      r.y = dpmpp_one(xv.y, mv.y, h1.y, h2.y, a, z.y);
      r.z = dpmpp_one(xv.z, mv.z, h1.z, h2.z, a, z.z);
      r.w = dpmpp_one(xv.w, mv.w, h1.w, h2.w, a, z.w);
      reinterpret_cast<float4*>(xn)[i] = r;
      reinterpret_cast<float4*>(d_out)[i] = z;
    } else {
      float z;
      const float r = dpmpp_one(x[i], __ldg(mo + i), d1 ? __ldg(d1 + i) : 0.f, d2 ? d2[i] : 0.f, a, z);
      xn[i] = r;
      d_out[i] = z;
    }
  }
  if (VEC == 4) {      // scalar tail: the last n % 4 elements
    const long i = items * 4 + tid;
    if (i < n) {
      float z;
      const float r = dpmpp_one(x[i], __ldg(mo + i), d1 ? __ldg(d1 + i) : 0.f, d2 ? d2[i] : 0.f, a, z);
      xn[i] = r;
      d_out[i] = z;
    }
  }
}

struct DdpmArgs {
  float coef1, coef2, sigma;
};

__device__ __forceinline__ float ddpm_one(float x, float mo, float nz, bool has_noise, const DdpmArgs& a, float& x0o) {
  const float x0 = clamp1(mo);
  x0o = x0;
  float r = __fadd_rn(__fmul_rn(a.coef1, x0), __fmul_rn(a.coef2, x));
  if (has_noise) r = __fadd_rn(r, __fmul_rn(a.sigma, nz));
  return r;
}

template <int VEC>
__global__ void __launch_bounds__(256) ddpm_kernel(const float* __restrict__ x, const float* __restrict__ mo,
                                                   const float* __restrict__ noise, float* __restrict__ xn,
                                                   float* __restrict__ x0_out, long n, DdpmArgs a) {
  const long items = n / VEC;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < items; i += (long)gridDim.x * blockDim.x) {
    if (VEC == 4) {
      const float4 xv = reinterpret_cast<const float4*>(x)[i];
      const float4 mv = __ldg(reinterpret_cast<const float4*>(mo) + i);
      float4 nv = make_float4(0.f, 0.f, 0.f, 0.f);
      if (noise) nv = __ldg(reinterpret_cast<const float4*>(noise) + i);
      float4 r, z;
      r.x = ddpm_one(xv.x, mv.x, nv.x, noise != nullptr, a, z.x);
      r.y = ddpm_one(xv.y, mv.y, nv.y, noise != nullptr, a, z.y);
      r.z = ddpm_one(xv.z, mv.z, nv.z, noise != nullptr, a, z.z);
      r.w = ddpm_one(xv.w, mv.w, nv.w, noise != nullptr, a, z.w);
      reinterpret_cast<float4*>(xn)[i] = r;
      if (x0_out) reinterpret_cast<float4*>(x0_out)[i] = z;
    } else {
      float z;
      const float r = ddpm_one(x[i], __ldg(mo + i), noise ? __ldg(noise + i) : 0.f, noise != nullptr, a, z);
      xn[i] = r;
      if (x0_out) x0_out[i] = z;
    }
  }
}

constexpr int kMseThreads = 256;

int mse_grid(long total) {
  long blocks = (total + kMseThreads * 4 - 1) / (kMseThreads * 4);
  const long cap = (long)FD_NUM_SMS * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

__global__ void __launch_bounds__(kMseThreads) nan_mse_fwd_kernel(const float* __restrict__ pred,
                                                                  const float* __restrict__ target,
                                                                  float* __restrict__ partials, int B, long CHW,
                                                                  long pred_bstride, long target_bstride) {
  __shared__ float red[2 * 32];
  float s[2] = {0.f, 0.f};
  const long total = (long)B * CHW;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long b = i / CHW, r = i % CHW;
    const float p = __ldg(pred + b * pred_bstride + r), q = __ldg(target + b * target_bstride + r);
    if (p == p && q == q) {
      const float d = p - q;
      s[0] += d * d;
      s[1] += 1.f;
    }
  }
  fd_block_sum<2>(s, red);
  if (threadIdx.x == 0) {
    partials[blockIdx.x * 2 + 0] = s[0];
    partials[blockIdx.x * 2 + 1] = s[1];
  }
}

// sums[0] = sum of squared errors, sums[1] = count, sums[2] = mean (NaN when count == 0, like nanmean of empty)
__global__ void __launch_bounds__(256) nan_mse_finalize_kernel(const float* __restrict__ partials, int nblocks,
                                                               float* __restrict__ sums) {
  __shared__ double sh[2][256];
  double a0 = 0.0, a1 = 0.0;
  for (int k = threadIdx.x; k < nblocks; k += 256) {
    a0 += (double)partials[2 * k];
    a1 += (double)partials[2 * k + 1];
  }
  sh[0][threadIdx.x] = a0;
  sh[1][threadIdx.x] = a1;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      sh[0][threadIdx.x] += sh[0][threadIdx.x + o];
      sh[1][threadIdx.x] += sh[1][threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    sums[0] = (float)sh[0][0];
    sums[1] = (float)sh[1][0];
    sums[2] = (float)(sh[0][0] / sh[1][0]);
  }
}

__global__ void __launch_bounds__(256) nan_mse_bwd_kernel(const float* __restrict__ pred,
                                                          const float* __restrict__ target,
                                                          const float* __restrict__ sums, float upstream,
                                                          float* __restrict__ gpred, int B, long CHW,
                                                          long pred_bstride, long target_bstride, long gpred_bstride) {
  const float gs = 2.f * upstream / __ldg(sums + 1);
  const long total = (long)B * CHW;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long b = i / CHW, r = i % CHW;
    const float p = __ldg(pred + b * pred_bstride + r), q = __ldg(target + b * target_bstride + r);
    gpred[b * gpred_bstride + r] = (p == p && q == q) ? gs * (p - q) : 0.f;
  }
}

}  // namespace

extern "C" {

int fd_q_sample(const float* x0, const float* noise, const int64_t* t, const float* sqrt_ac, const float* sqrt_1mac,
                float* out, int B, long per_sample, void* stream) {
  FD_REQUIRE(x0 && noise && t && sqrt_ac && sqrt_1mac && out && B > 0 && per_sample > 0, "q_sample: bad argument");
  q_sample_kernel<<<egrid((long)B * per_sample), 256, 0, (cudaStream_t)stream>>>(x0, noise, t, sqrt_ac, sqrt_1mac, out,
                                                                                  B, per_sample);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

static bool aligned16(const void* p) { return p == nullptr || (((uintptr_t)p) & 15) == 0; }

int fd_ddim_step(const float* x, const float* model_out, const float* noise, float* x_next, float* x0_out, long n,
                 float recip, float recipm1, float sqrt_alpha_next, float c, float sigma, int last, void* stream) {
  FD_REQUIRE(x && model_out && x_next && n > 0, "ddim_step: bad argument");
  FD_REQUIRE(noise != nullptr || sigma == 0.f || last, "ddim_step: sigma != 0 needs a noise tensor");
  DdimArgs a{recip, recipm1, sqrt_alpha_next, c, sigma, last};
  if (last || sigma == 0.f) noise = nullptr;   // sigma*noise == +-0 leaves the fp32 sum unchanged
  const bool v4 = (n % 4 == 0) && aligned16(x) && aligned16(model_out) && aligned16(noise) && aligned16(x_next) &&
                  aligned16(x0_out);
  if (v4)
    ddim_kernel<4><<<egrid(n / 4), 256, 0, (cudaStream_t)stream>>>(x, model_out, noise, x_next, x0_out, n, a);
  else
    ddim_kernel<1><<<egrid(n), 256, 0, (cudaStream_t)stream>>>(x, model_out, noise, x_next, x0_out, n, a);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_dpmpp_step(const float* x, const float* model_out, const float* d_hist1, const float* d_hist2, float* x_next,
                  float* d_out, long n, float cx, float c0, float c1, float c2, int last, void* stream) {
  FD_REQUIRE(x && model_out && x_next && d_out && n > 0, "dpmpp_step: bad argument");
  if (last) c1 = c2 = 0.f;
  FD_REQUIRE(c1 == 0.f || d_hist1 != nullptr, "dpmpp_step: c1 != 0 needs d_hist1");
  FD_REQUIRE(c2 == 0.f || d_hist2 != nullptr, "dpmpp_step: c2 != 0 needs d_hist2");
  if (c1 == 0.f) d_hist1 = nullptr;    // unused history is not read
  if (c2 == 0.f) d_hist2 = nullptr;
  FD_REQUIRE(d_out != x_next && d_out != d_hist1 && d_out != x && x_next != d_hist1 && x_next != d_hist2,
             "dpmpp_step: only x_next == x and d_out == d_hist2 may alias");
  DpmppArgs a{cx, c0, c1, c2, last};
  const bool v4 = aligned16(x) && aligned16(model_out) && aligned16(d_hist1) && aligned16(d_hist2) &&
                  aligned16(x_next) && aligned16(d_out);
  if (v4)
    dpmpp_kernel<4><<<egrid(n / 4), 256, 0, (cudaStream_t)stream>>>(x, model_out, d_hist1, d_hist2, x_next, d_out, n,
                                                                  a);
  else
    dpmpp_kernel<1><<<egrid(n), 256, 0, (cudaStream_t)stream>>>(x, model_out, d_hist1, d_hist2, x_next, d_out, n, a);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_ddpm_step(const float* x, const float* model_out, const float* noise, float* x_next, float* x0_out, long n,
                 float coef1, float coef2, float sigma, void* stream) {
  FD_REQUIRE(x && model_out && x_next && n > 0, "ddpm_step: bad argument");
  DdpmArgs a{coef1, coef2, sigma};
  const bool v4 = (n % 4 == 0) && aligned16(x) && aligned16(model_out) && aligned16(noise) && aligned16(x_next) &&
                  aligned16(x0_out);
  if (v4)
    ddpm_kernel<4><<<egrid(n / 4), 256, 0, (cudaStream_t)stream>>>(x, model_out, noise, x_next, x0_out, n, a);
  else
    ddpm_kernel<1><<<egrid(n), 256, 0, (cudaStream_t)stream>>>(x, model_out, noise, x_next, x0_out, n, a);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

size_t fd_nan_mse_workspace_floats(int B, int C, int HW) { return (size_t)mse_grid((long)B * C * HW) * 2; }

int fd_nan_mse_fwd(const float* pred, const float* target, float* sums, float* partials, int B, int C, int HW,
                   long pred_bstride, long target_bstride, void* stream) {
  FD_REQUIRE(pred && target && sums && partials && B > 0 && C > 0 && HW > 0, "nan_mse_fwd: bad argument");
  const long CHW = (long)C * HW;
  const int grid = mse_grid((long)B * CHW);
  nan_mse_fwd_kernel<<<grid, kMseThreads, 0, (cudaStream_t)stream>>>(pred, target, partials, B, CHW, pred_bstride,
                                                                      target_bstride);
  FD_LAUNCH_CHECK();
  nan_mse_finalize_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(partials, grid, sums);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_nan_mse_bwd(const float* pred, const float* target, const float* sums, float upstream, float* gpred, int B,
                   int C, int HW, long pred_bstride, long target_bstride, long gpred_bstride, void* stream) {
  FD_REQUIRE(pred && target && sums && gpred && B > 0 && C > 0 && HW > 0, "nan_mse_bwd: bad argument");
  const long CHW = (long)C * HW;
  nan_mse_bwd_kernel<<<egrid((long)B * CHW), 256, 0, (cudaStream_t)stream>>>(pred, target, sums, upstream, gpred, B,
                                                                             CHW, pred_bstride, target_bstride,
                                                                             gpred_bstride);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

}  // extern "C"
