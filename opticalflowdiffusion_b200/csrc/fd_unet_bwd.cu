// HBM-bound pieces of the UNet BACKWARD pass (the autograd graph of denoising_diffusion.py:81-417 that
// `loss.backward()` walks in the reference's training_step, flow_diffuser.py:217-235) on bf16 NHWC
// activations: GroupNorm + scale/shift + SiLU backward, channel-LayerNorm backward, nearest-upsample
// backward, final 1x1 conv backward, bias gradients, weight (un)packing for dgrad / wgrad including the
// weight-standardisation backward, the time-embedding MLP backward, and the fused clip + Adam update.
// Activation kernels move 16 bytes (8 channels) per access like their forward counterparts; per-channel
// parameter gradients are reduced in registers -> shared memory -> one fp32 atomic per block and channel.
#include "fd_common.cuh"

namespace {

int egrid(long items, int threads, int per_sm = 16) {
  long blocks = (items + threads - 1) / threads;
  const long cap = (long)FD_NUM_SMS * per_sm;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 p = fd_unpack_bf16(w[e]);
    f[2 * e] = p.x;
    f[2 * e + 1] = p.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 o;
  o.x = fd_pack_bf16(f[0], f[1]);
  o.y = fd_pack_bf16(f[2], f[3]);
  o.z = fd_pack_bf16(f[4], f[5]);
  o.w = fd_pack_bf16(f[6], f[7]);
  return o;
}

// ---------------------------------------------------------------------------------------------
// GroupNorm(8) + (scale+1, shift) + SiLU backward  (Block.forward :181-187).
//   forward:  xh = (h - mean_g) rstd_g ; y = xh gamma + beta ; z = y (scale+1) + shift ; a = silu(z)
//   pass 1 (reduce):  per (n, c):  S0 = sum dz, S1 = sum dz*h, S2 = sum h      with dz = da * silu'(z)
//   pass 2 (finalize, tiny): parameter gradients, per-(n,g) means of dxh and dxh*xh, conv-bias gradient
//   pass 3 (apply):   dh = P_c dz + Q_g h + R_g
// z is recomputed from h with the forward's folded coefficients (a_c h + b_c); nothing but h is saved.
// ---------------------------------------------------------------------------------------------
struct GnCoef {
  float a[8], b[8];
};

__device__ __forceinline__ void gn_fold(const double* __restrict__ stats, const float* __restrict__ gamma,
                                        const float* __restrict__ beta, const float* __restrict__ scale_shift,
                                        long ss_stride, int n, int chunk, int C, long HW, float eps, GnCoef& k) {
  // C % 64 == 0, so the channels-per-group count is a multiple of 8 and the thread's 8 channels share ONE group: the
  // double-precision mean / rstd are computed once per thread.  (Per channel, i.e. 8 x 3 double divisions / square roots per
  // thread, this prologue was ~20 us of every launch -- measured: 46 us for a 72 MB reduce at 46x96x512.)
  const int cpg = C >> 3;
  const double cnt = (double)HW * cpg;
  const int g = (chunk * 8) / cpg;
  const double s = stats[((long)n * 8 + g) * 2], ss = stats[((long)n * 8 + g) * 2 + 1];
  const double mean = s / cnt;
  double var = ss / cnt - mean * mean;
  if (var < 0.0) var = 0.0;
  const float rstd = (float)(1.0 / sqrt(var + (double)eps));
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = chunk * 8 + j;
    float ga = __ldg(gamma + c) * rstd;
    float be = __ldg(beta + c) - (float)mean * ga;
    if (scale_shift != nullptr) {
      const float sc = __ldg(scale_shift + (long)n * ss_stride + c) + 1.f;
      const float sh = __ldg(scale_shift + (long)n * ss_stride + C + c);
      ga *= sc;
      be = be * sc + sh;
    }
    k.a[j] = ga;
    k.b[j] = be;
  }
}

// d/dz silu(z) = s + z s (1 - s) with s = sigmoid(z) = 0.5 tanh(z / 2) + 0.5: ONE MUFU op (tanh.approx, 2^-11 relative)
// instead of ex2 + rcp -- the two GroupNorm backward passes were XU / issue bound (ncu: XU 42 %, issue 60-65 %)
__device__ __forceinline__ float silu_grad(float z) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * z));
  const float sg = fmaf(t, 0.5f, 0.5f);
  return fmaf(z * sg, 1.f - sg, sg);
}

__global__ void __launch_bounds__(256, 2) gn_bwd_reduce_kernel(const __nv_bfloat16* __restrict__ h,
                                                            const __nv_bfloat16* __restrict__ da,
                                                            const double* __restrict__ stats,
                                                            const float* __restrict__ gamma, const float* __restrict__ beta,
                                                            const float* __restrict__ scale_shift, long ss_stride,
                                                            float* __restrict__ partial /* [N][gridDim.x][C][3] */, long HW,
                                                            int C, float eps) {
  extern __shared__ float s_acc[];      // [rows of the block][C][3]: fixed-order reduction, no atomics (run-to-run stable)
  const int n = blockIdx.y;
  const int chunks = C >> 3;
  const int chunk = threadIdx.x % chunks;
  const int prow = threadIdx.x / chunks;
  const int ppb = blockDim.x / chunks;
  GnCoef k;
  gn_fold(stats, gamma, beta, scale_shift, ss_stride, n, chunk, C, HW, eps, k);
  float s0[8], s1[8], s2[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s0[j] = s1[j] = s2[j] = 0.f;
  const long base = (long)n * HW;
  constexpr int U = 4;
  const long stride = (long)gridDim.x * ppb;
  for (long p0 = (long)blockIdx.x * ppb + prow; p0 < HW; p0 += stride * U) {
    uint4 hv[U], dv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long p = p0 + u * stride;
      if (p < HW) {
        const long off = (base + p) * C + chunk * 8;
        hv[u] = __ldcs(reinterpret_cast<const uint4*>(h + off));
        dv[u] = __ldcs(reinterpret_cast<const uint4*>(da + off));
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (p0 + u * stride >= HW) break;
      float hf[8], df[8];
      unpack8(hv[u], hf);
      unpack8(dv[u], df);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float dz = df[j] * silu_grad(k.a[j] * hf[j] + k.b[j]);
        s0[j] += dz;
        s1[j] += dz * hf[j];
        s2[j] += hf[j];
      }
    }
  }
  float* mine = s_acc + (long)prow * C * 3;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = chunk * 8 + j;
    mine[c * 3 + 0] = s0[j];
    mine[c * 3 + 1] = s1[j];
    mine[c * 3 + 2] = s2[j];
  }
  __syncthreads();
  float* out = partial + ((long)n * gridDim.x + blockIdx.x) * C * 3;
  for (int i = threadIdx.x; i < C * 3; i += blockDim.x) {
    float v = 0.f;
    for (int r = 0; r < ppb; ++r) v += s_acc[(long)r * C * 3 + i];
    out[i] = v;
  }
}

// one block per (sample, group): blockDim = (C / 8 channels of the group, S slices of the reduce kernel's blocks).  The first
// version ran one block per SAMPLE with 1024 / C slices: for C = 512 a thread walked 75 partial blocks (47 us per launch,
// 12-47 us over the 38 GroupNorms of a step, pure load latency on 8 SMs); per-group blocks give 8x the blocks and up to
// 32 slices whatever C is.
__global__ void __launch_bounds__(1024) gn_bwd_finalize_kernel(const float* __restrict__ partial, int nblocks,
                                                               const double* __restrict__ stats,
                                                               const float* __restrict__ gamma, const float* __restrict__ beta,
                                                               const float* __restrict__ scale_shift, long ss_stride,
                                                               float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                               float* __restrict__ dss, float* __restrict__ dbias,
                                                               float* __restrict__ coef /* [N][8][2] */, long HW, int C,
                                                               float eps) {
  __shared__ float s_g[2];
  __shared__ float s_c[128][2];            // channels of the group (C <= 1024)
  __shared__ float s_p[1024 * 3];          // [blockDim.y slices][C / 8][3]
  const int n = blockIdx.x, g = blockIdx.y;
  const int cpg = C >> 3;
  const int cl = threadIdx.x, c = g * cpg + cl;
  const double cnt = (double)HW * cpg;
  const double s = stats[((long)n * 8 + g) * 2], ss = stats[((long)n * 8 + g) * 2 + 1];
  const double mean_d = s / cnt;
  double var = ss / cnt - mean_d * mean_d;
  if (var < 0.0) var = 0.0;
  const float rstd = (float)(1.0 / sqrt(var + (double)eps));
  const float mean = (float)mean_d;
  // Sum of the reduce kernel's per-block partials in a FIXED order (run-to-run stable), spread over blockDim.y slices of
  // blocks with four independent accumulators each: the loop is pure load latency.
  float S0, S1, S2;
  {
    constexpr int U = 4;
    float a0[U], a1[U], a2[U];
#pragma unroll
    for (int u = 0; u < U; ++u) a0[u] = a1[u] = a2[u] = 0.f;
    const float* pn = partial + ((long)n * nblocks * C + c) * 3;
    const int S = blockDim.y, sl = threadIdx.y;
    int bb = sl;
    for (; bb + (U - 1) * S < nblocks; bb += U * S) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float* pb = pn + (long)(bb + u * S) * C * 3;
        a0[u] += pb[0];
        a1[u] += pb[1];
        a2[u] += pb[2];
      }
    }
    for (; bb < nblocks; bb += S) {
      const float* pb = pn + (long)bb * C * 3;
      a0[0] += pb[0];
      a1[0] += pb[1];
      a2[0] += pb[2];
    }
    float* mine = s_p + ((long)sl * cpg + cl) * 3;
    mine[0] = (a0[0] + a0[1]) + (a0[2] + a0[3]);
    mine[1] = (a1[0] + a1[1]) + (a1[2] + a1[3]);
    mine[2] = (a2[0] + a2[1]) + (a2[2] + a2[3]);
    __syncthreads();
    S0 = S1 = S2 = 0.f;
    if (sl == 0) {
      for (int q = 0; q < S; ++q) {
        const float* o = s_p + ((long)q * cpg + cl) * 3;
        S0 += o[0];
        S1 += o[1];
        S2 += o[2];
      }
    }
  }
  const bool lead = threadIdx.y == 0;                  // slice 0 holds the full sums and does the rest of the (tiny) work
  const float Sx = rstd * (S1 - mean * S0);            // sum dz * xh
  const float ga = gamma[c], be = beta[c];
  const float sc = scale_shift != nullptr ? scale_shift[(long)n * ss_stride + c] + 1.f : 1.f;
  if (lead) {
    atomicAdd(dgamma + c, sc * Sx);
    atomicAdd(dbeta + c, sc * S0);
    if (dss != nullptr) {
      dss[(long)n * ss_stride + c] = ga * Sx + be * S0;  // d scale = sum dz * y
      dss[(long)n * ss_stride + C + c] = S0;             // d shift
    }
    s_c[cl][0] = sc * ga * S0;                           // dxh summed over the pixels of this channel
    s_c[cl][1] = sc * ga * Sx;                           // ... dxh * xh
  }
  __syncthreads();
  if (lead && cl == 0) {                                 // group sums in channel order
    float a = 0.f, b = 0.f;
    for (int i = 0; i < cpg; ++i) {
      a += s_c[i][0];
      b += s_c[i][1];
    }
    s_g[0] = a;
    s_g[1] = b;
  }
  __syncthreads();
  if (!lead) return;
  const float m1 = s_g[0] / (float)cnt, m2 = s_g[1] / (float)cnt;
  const float Q = -rstd * rstd * m2;
  const float R = -rstd * m1 - Q * mean;
  if (cl == 0) {
    coef[((long)n * 8 + g) * 2] = Q;
    coef[((long)n * 8 + g) * 2 + 1] = R;
  }
  if (dbias != nullptr) atomicAdd(dbias + c, rstd * sc * ga * S0 + Q * S2 + R * (float)HW);   // sum over pixels of dh
}

__global__ void __launch_bounds__(256, 3) gn_bwd_apply_kernel(const __nv_bfloat16* __restrict__ h,
                                                           const __nv_bfloat16* __restrict__ da,
                                                           const double* __restrict__ stats, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta,
                                                           const float* __restrict__ scale_shift, long ss_stride,
                                                           const float* __restrict__ coef, __nv_bfloat16* __restrict__ dh,
                                                           long HW, int C, float eps) {
  const int n = blockIdx.y;
  const int chunks = C >> 3;
  const int chunk = threadIdx.x % chunks;
  const int prow = threadIdx.x / chunks;
  const int ppb = blockDim.x / chunks;
  const int cpg = C >> 3;
  GnCoef k;
  gn_fold(stats, gamma, beta, scale_shift, ss_stride, n, chunk, C, HW, eps, k);
  // C % 64 == 0 -> channels-per-group is a multiple of 8: the thread's 8 channels share one group
  const int grp = (chunk * 8) / cpg;
  const float Q = coef[((long)n * 8 + grp) * 2], R = coef[((long)n * 8 + grp) * 2 + 1];
  // P_c = rstd (scale+1) gamma = k.a (the folded forward slope)
  const long base = (long)n * HW;
  constexpr int U = 4;
  const long stride = (long)gridDim.x * ppb;
  for (long p0 = (long)blockIdx.x * ppb + prow; p0 < HW; p0 += stride * U) {
    uint4 hv[U], dv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long p = p0 + u * stride;
      if (p < HW) {
        const long off = (base + p) * C + chunk * 8;
        hv[u] = __ldcs(reinterpret_cast<const uint4*>(h + off));
        dv[u] = __ldcs(reinterpret_cast<const uint4*>(da + off));
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long p = p0 + u * stride;
      if (p >= HW) break;
      float hf[8], df[8], o[8];
      unpack8(hv[u], hf);
      unpack8(dv[u], df);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float dz = df[j] * silu_grad(k.a[j] * hf[j] + k.b[j]);
        o[j] = k.a[j] * dz + Q * hf[j] + R;
      }
      *reinterpret_cast<uint4*>(dh + (base + p) * C + chunk * 8) = pack8(o);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// channel LayerNorm backward (:116-125):  y = xh g ;  dx = rstd (dxh - mean(dxh) - xh mean(dxh xh)) (+ add),
// dg[c] += sum_px dy xh.  Same thread mapping as the forward kernel.
// ---------------------------------------------------------------------------------------------
template <int LANES, int CHUNKS>
__global__ void __launch_bounds__(256) chan_ln_bwd_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ g,
                                                          const __nv_bfloat16* __restrict__ dy,
                                                          const __nv_bfloat16* __restrict__ add,
                                                          __nv_bfloat16* __restrict__ dx, float* __restrict__ dg, long npix,
                                                          float eps) {
  constexpr int C = LANES * CHUNKS * 8;
  __shared__ float s_dg[C];
  for (int i = threadIdx.x; i < C; i += blockDim.x) s_dg[i] = 0.f;
  __syncthreads();
  const int sub = threadIdx.x % LANES;
  const long gid = ((long)blockIdx.x * blockDim.x + threadIdx.x) / LANES;
  const long gstride = ((long)gridDim.x * blockDim.x) / LANES;
  float gain[CHUNKS][8], acc[CHUNKS][8];
#pragma unroll
  for (int k = 0; k < CHUNKS; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      gain[k][j] = __ldg(g + (k * LANES + sub) * 8 + j);
      acc[k][j] = 0.f;
    }
  const long iters = (npix + gstride - 1) / gstride;
  for (long it = 0; it < iters; ++it) {
    const long p = gid + it * gstride;
    const bool valid = p < npix;
    float v[CHUNKS][8], d[CHUNKS][8];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < CHUNKS; ++k) {
      uint4 xv = make_uint4(0, 0, 0, 0), dv = make_uint4(0, 0, 0, 0);
      if (valid) {
        xv = __ldg(reinterpret_cast<const uint4*>(x + p * C + (k * LANES + sub) * 8));
        dv = __ldg(reinterpret_cast<const uint4*>(dy + p * C + (k * LANES + sub) * 8));
      }
      unpack8(xv, v[k]);
      unpack8(dv, d[k]);
#pragma unroll
      for (int j = 0; j < 8; ++j) s += v[k][j];
    }
#pragma unroll
    for (int o = LANES / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s * (1.f / C);
    float ss = 0.f;
#pragma unroll
    for (int k = 0; k < CHUNKS; ++k)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        v[k][j] -= mean;
        ss += v[k][j] * v[k][j];
      }
#pragma unroll
    for (int o = LANES / 2; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const float rstd = rsqrtf(ss * (1.f / C) + eps);
    float m1 = 0.f, m2 = 0.f;
#pragma unroll
    for (int k = 0; k < CHUNKS; ++k)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        v[k][j] *= rstd;                              // xh
        acc[k][j] += d[k][j] * v[k][j];               // dg
        d[k][j] *= gain[k][j];                        // dxh
        m1 += d[k][j];
        m2 += d[k][j] * v[k][j];
      }
#pragma unroll
    for (int o = LANES / 2; o > 0; o >>= 1) {
      m1 += __shfl_xor_sync(0xffffffffu, m1, o);
      m2 += __shfl_xor_sync(0xffffffffu, m2, o);
    }
    m1 *= (1.f / C);
    m2 *= (1.f / C);
    if (valid) {
#pragma unroll
      for (int k = 0; k < CHUNKS; ++k) {
        const long off = p * C + (k * LANES + sub) * 8;
        float y[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = rstd * (d[k][j] - m1 - v[k][j] * m2);
        if (add != nullptr) {
          float af[8];
          unpack8(__ldg(reinterpret_cast<const uint4*>(add + off)), af);
#pragma unroll
          for (int j = 0; j < 8; ++j) y[j] += af[j];
        }
        *reinterpret_cast<uint4*>(dx + off) = pack8(y);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < CHUNKS; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) atomicAdd(&s_dg[(k * LANES + sub) * 8 + j], acc[k][j]);
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x) atomicAdd(dg + i, s_dg[i]);
}

// nearest 2x upsample backward (:91): dx[n,h,w,:] = sum of the 2x2 block of dy (N,2H,2W,C)
__global__ void __launch_bounds__(256) upsample2x_bwd_kernel(const uint4* __restrict__ dy, uint4* __restrict__ dx, long N,
                                                             int H, int W, int C8) {
  const long total = N * H * W * C8;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C8);
    long r = i / C8;
    const int w = (int)(r % W);
    r /= W;
    const int h = (int)(r % H);
    const long n = r / H;
    const long o = ((n * 2 * H + 2 * h) * 2 * W + 2 * w) * C8 + c;
    float a[8], b[8];
    unpack8(__ldcs(dy + o), a);
    unpack8(__ldcs(dy + o + C8), b);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] += b[j];
    unpack8(__ldcs(dy + o + (long)2 * W * C8), b);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] += b[j];
    unpack8(__ldcs(dy + o + (long)2 * W * C8 + C8), b);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] += b[j];
    dx[i] = pack8(a);
  }
}

// out = a + b (bf16, 16-byte granules): gradient accumulation where no producer epilogue can absorb it
__global__ void __launch_bounds__(256) add_bf16_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b,
                                                       uint4* __restrict__ out, long n16) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (long)gridDim.x * blockDim.x) {
    float x[8], y[8];
    unpack8(__ldcs(a + i), x);
    unpack8(__ldcs(b + i), y);
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] += y[j];
    out[i] = pack8(x);
  }
}

// bias gradient of a convolution: db[c] += sum over pixels of dy[p][c]   (bf16 [npix][C])
__global__ void __launch_bounds__(256) bias_grad_kernel(const __nv_bfloat16* __restrict__ dy, float* __restrict__ db, long npix,
                                                        int C) {
  extern __shared__ float s_acc[];      // [C]
  const int chunks = C >> 3;
  const int chunk = threadIdx.x % chunks;
  const int prow = threadIdx.x / chunks;
  const int ppb = blockDim.x / chunks;
  for (int i = threadIdx.x; i < C; i += blockDim.x) s_acc[i] = 0.f;
  __syncthreads();
  float s[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = 0.f;
  for (long p = (long)blockIdx.x * ppb + prow; p < npix; p += (long)gridDim.x * ppb) {
    float f[8];
    unpack8(__ldcs(reinterpret_cast<const uint4*>(dy + p * C + chunk * 8)), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] += f[j];
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) atomicAdd(&s_acc[chunk * 8 + j], s[j]);
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x) atomicAdd(db + i, s_acc[i]);
}

// final 1x1 conv backward (:361,417): dout fp32 NCHW (N,Cout<=4,HW), x bf16 (N,HW,64)
//   dx[p][c] = sum_o dout[o][p] w[o][c] ;  dw[o][c] += sum_p dout[o][p] x[p][c] ;  db[o] += sum_p dout[o][p]
__global__ void __launch_bounds__(256) final_conv_bwd_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w,
                                                             const float* __restrict__ dout, __nv_bfloat16* __restrict__ dx,
                                                             float* __restrict__ dw, float* __restrict__ db, int N, long HW,
                                                             int Cout) {
  constexpr int Cin = 64;
  __shared__ float s_dw[4 * Cin + 4];
  for (int i = threadIdx.x; i < 4 * Cin + 4; i += blockDim.x) s_dw[i] = 0.f;
  __syncthreads();
  const int chunk = threadIdx.x & 7;
  float wr[4][8], aw[4][8], ab[4];
#pragma unroll
  for (int o = 0; o < 4; ++o) {
    ab[o] = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      wr[o][j] = o < Cout ? __ldg(w + o * Cin + chunk * 8 + j) : 0.f;
      aw[o][j] = 0.f;
    }
  }
  const long total = (long)N * HW;
  for (long i = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 3; i < total; i += ((long)gridDim.x * blockDim.x) >> 3) {
    const long n = i / HW, p = i - n * HW;
    float d[4];
#pragma unroll
    for (int o = 0; o < 4; ++o) d[o] = o < Cout ? __ldg(dout + (n * Cout + o) * HW + p) : 0.f;
    float xf[8], y[8];
    unpack8(__ldcs(reinterpret_cast<const uint4*>(x + i * Cin + chunk * 8)), xf);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      y[j] = 0.f;
#pragma unroll
      for (int o = 0; o < 4; ++o) {
        y[j] += d[o] * wr[o][j];
        aw[o][j] += d[o] * xf[j];
      }
    }
#pragma unroll
    for (int o = 0; o < 4; ++o) ab[o] += d[o];
    *reinterpret_cast<uint4*>(dx + i * Cin + chunk * 8) = pack8(y);
  }
#pragma unroll
  for (int o = 0; o < 4; ++o) {
#pragma unroll
    for (int j = 0; j < 8; ++j) atomicAdd(&s_dw[o * Cin + chunk * 8 + j], aw[o][j]);
    if (chunk == 0) atomicAdd(&s_dw[4 * Cin + o], ab[o]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < Cout * Cin; i += blockDim.x) atomicAdd(dw + i, s_dw[i]);
  if (threadIdx.x < Cout) atomicAdd(db + threadIdx.x, s_dw[4 * Cin + threadIdx.x]);
}

// ---------------------------------------------------------------------------------------------
// dgrad weights: the forward's packed bf16 [Cout][T*Cin] -> [Cin][T*Cout] with the taps reversed, so that the data
// gradient is the SAME implicit-GEMM convolution run on dy:  wd[ci][(T-1-tap)*Cout + co] = wf[co][tap*Cin + ci].
// 32x32 shared-memory transpose per tap.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void prep_weight_dgrad_body(const __nv_bfloat16* __restrict__ wf, __nv_bfloat16* __restrict__ wd,
                                                       int Cout, int Cin, int T, int bx, int by, int tap) {
  __shared__ __nv_bfloat16 tile[32][34];
  const int ci0 = bx * 32, co0 = by * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int co = co0 + r, ci = ci0 + tx;
    if (co < Cout && ci < Cin) tile[r][tx] = wf[(long)co * T * Cin + (long)tap * Cin + ci];
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int ci = ci0 + r, co = co0 + tx;
    if (co < Cout && ci < Cin) wd[(long)ci * T * Cout + (long)(T - 1 - tap) * Cout + co] = tile[tx][r];
  }
}

__global__ void __launch_bounds__(256) prep_weight_dgrad_kernel(const __nv_bfloat16* __restrict__ wf,
                                                                __nv_bfloat16* __restrict__ wd, int Cout, int Cin, int T) {
  prep_weight_dgrad_body(wf, wd, Cout, Cin, T, blockIdx.x, blockIdx.y, blockIdx.z);
}

__device__ __forceinline__ int batch_find_layer(const int* __restrict__ blk_start, int n_layers, int b) {
  int lo = 0, hi = n_layers;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (blk_start[mid] <= b) lo = mid; else hi = mid;
  }
  return lo;
}

// every layer's dgrad weights in one launch (table record: packed, wd, -, Cout, Cin, taps)
__global__ void __launch_bounds__(256) prep_weight_dgrad_batch_kernel(const long long* __restrict__ table,
                                                                      const int* __restrict__ blk_start, int n_layers) {
  const int l = batch_find_layer(blk_start, n_layers, (int)blockIdx.x);
  const long long* r = table + (long)l * 8;
  const int Cout = (int)r[3], Cin = (int)r[4], T = (int)r[5];
  int b = (int)blockIdx.x - blk_start[l];
  const int nx = (Cin + 31) / 32, ny = (Cout + 31) / 32;
  const int bx = b % nx;
  b /= nx;
  prep_weight_dgrad_body(reinterpret_cast<const __nv_bfloat16*>(r[0]), reinterpret_cast<__nv_bfloat16*>(r[1]), Cout, Cin, T, bx,
                         b % ny, b / ny);
}

// ---------------------------------------------------------------------------------------------
// wgrad unpacking + weight-standardisation backward (:106-114).  g: fp32 packed [Cout][Kp] (fd_conv_wgrad order),
// w: the fp32 parameter [Cout][Cin][KH][KW]; dw (same layout) += the parameter gradient.
//   wt = (w - mean) r ;  dw = r (g - mean(g) - wt mean(g wt))      one block per output channel
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void prep_weight_bwd_body(const float* __restrict__ g, const float* __restrict__ w,
                                                     float* __restrict__ dw, int Cin, int KH, int KW, int kind,
                                                     int standardize, float eps, int Kpacked, int o) {
  __shared__ float red[64];
  __shared__ float s_a, s_b;
  const int n = Cin * KH * KW;
  const float* wo = w + (long)o * n;
  const float* go = g + (long)o * Kpacked;
  float* dwo = dw + (long)o * n;
  auto kidx = [&](int i) {
    const int kx = i % KW;
    const int ky = (i / KW) % KH;
    const int ci = i / (KW * KH);
    if (kind == 0) return (ky * KW + kx) * Cin + ci;
    if (kind == 1) return (ci & 3) * (Cin / 4) + (ci >> 2);
    if (kind == 3) return (ky * KW + kx) * 64 + ci;
    return ky * 64 + kx * Cin + ci;
  };
  if (!standardize) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) dwo[i] += go[kidx(i)];
    return;
  }
  float s[1] = {0.f};
  for (int i = threadIdx.x; i < n; i += blockDim.x) s[0] += wo[i];
  fd_block_sum<1>(s, red);
  if (threadIdx.x == 0) s_a = s[0] / (float)n;
  __syncthreads();
  const float mean = s_a;
  float v[1] = {0.f};
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float d = wo[i] - mean;
    v[0] += d * d;
  }
  fd_block_sum<1>(v, red);
  if (threadIdx.x == 0) s_b = rsqrtf(v[0] / (float)n + eps);
  __syncthreads();
  const float rstd = s_b;
  float q[2] = {0.f, 0.f};
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float gi = go[kidx(i)];
    q[0] += gi;
    q[1] += gi * (wo[i] - mean) * rstd;
  }
  fd_block_sum<2>(q, red);
  __syncthreads();
  if (threadIdx.x == 0) {
    s_a = q[0] / (float)n;
    s_b = q[1] / (float)n;
  }
  __syncthreads();
  const float mg = s_a, mgw = s_b;
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    dwo[i] += rstd * (go[kidx(i)] - mg - (wo[i] - mean) * rstd * mgw);
}

__global__ void __launch_bounds__(256) prep_weight_bwd_kernel(const float* __restrict__ g, const float* __restrict__ w,
                                                              float* __restrict__ dw, int Cout, int Cin, int KH, int KW,
                                                              int kind, int standardize, float eps, int Kpacked) {
  prep_weight_bwd_body(g, w, dw, Cin, KH, KW, kind, standardize, eps, Kpacked, blockIdx.x);
}

// every conv's wgrad unpacking + weight-standardisation backward in one launch (table record: g, w, dw, Cout, Cin, KH, KW,
// kind | standardize << 8)
__global__ void __launch_bounds__(256) prep_weight_bwd_batch_kernel(const long long* __restrict__ table,
                                                                    const int* __restrict__ blk_start, int n_layers, float eps) {
  const int l = batch_find_layer(blk_start, n_layers, (int)blockIdx.x);
  const long long* r = table + (long)l * 8;
  const int Cin = (int)r[4], KH = (int)r[5], KW = (int)r[6], kind = (int)(r[7] & 0xff), ws = (int)((r[7] >> 8) & 1);
  const int Kp = kind == 2 ? KH * 64 : (kind == 3 ? KH * KW * 64 : Cin * KH * KW);
  prep_weight_bwd_body(reinterpret_cast<const float*>(r[0]), reinterpret_cast<const float*>(r[1]), reinterpret_cast<float*>(r[2]),
                       Cin, KH, KW, kind, ws, eps, Kp, (int)blockIdx.x - blk_start[l]);
}

// ---------------------------------------------------------------------------------------------
// small dense layers of the time path (:319-324 time_mlp, :193-196 ResnetBlock.mlp), fp32, batch <= a few dozen.
//   lin_bwd_w:  dW[j][k] += sum_b dY[b][j] act(X[b][k]) ;  db[j] += sum_b dY[b][j]
//   lin_bwd_x:  dX[b][k]  = act'(A[b][k]) sum_j dY[b][j] W[j][k]
// act: 0 identity, 1 SiLU, 2 GELU(erf)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float act_fwd(float x, int act) {
  if (act == 1) return x / (1.f + expf(-x));
  if (act == 2) return 0.5f * x * (1.f + erff(x * 0.70710678118654752440f));
  return x;
}
__device__ __forceinline__ float act_bwd(float x, int act) {
  if (act == 1) {
    const float sg = 1.f / (1.f + expf(-x));
    return sg * (1.f + x * (1.f - sg));
  }
  if (act == 2)
    return 0.5f * (1.f + erff(x * 0.70710678118654752440f)) + x * 0.3989422804014327f * expf(-0.5f * x * x);
  return 1.f;
}

__global__ void __launch_bounds__(256) lin_bwd_w_kernel(const float* __restrict__ dY, long dy_stride,
                                                        const float* __restrict__ X, long x_stride, float* __restrict__ dW,
                                                        float* __restrict__ db, int B, int J, int K, int act) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long)J * K) return;
  const int j = (int)(i / K), k = (int)(i % K);
  float acc = 0.f, accb = 0.f;
  for (int b = 0; b < B; ++b) {
    const float d = dY[(long)b * dy_stride + j];
    acc += d * act_fwd(X[(long)b * x_stride + k], act);
    accb += d;
  }
  dW[i] += acc;
  if (k == 0 && db != nullptr) db[j] += accb;
}

// block = (b, 32 consecutive k); 8 j-lanes x 32 k: coalesced rows of W, then a shared-memory reduction over the j-lanes
__global__ void __launch_bounds__(256) lin_bwd_x_kernel(const float* __restrict__ dY, long dy_stride,
                                                        const float* __restrict__ W, const float* __restrict__ A,
                                                        long a_stride, float* __restrict__ dX, long dx_stride, int B, int J,
                                                        int K, int act) {
  __shared__ float red[8][33];
  const int kb = blockIdx.x, b = blockIdx.y;
  const int kl = threadIdx.x & 31, jl = threadIdx.x >> 5;
  const int k = kb * 32 + kl;
  float acc = 0.f;
  if (k < K)
    for (int j = jl; j < J; j += 8) acc += __ldg(dY + (long)b * dy_stride + j) * __ldg(W + (long)j * K + k);
  red[jl][kl] = acc;
  __syncthreads();
  if (jl == 0 && k < K) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += red[i][kl];
    dX[(long)b * dx_stride + k] = s * act_bwd(A[(long)b * a_stride + k], act);
  }
}

// ---------------------------------------------------------------------------------------------
// optimiser: global gradient-norm clip (Lightning gradient_clip_val, exp_base.py:192,205) + torch.optim.Adam with
// L2-in-gradient weight decay (flow_diffuser.py:129-134), one pass over flat fp32 buffers.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sumsq_kernel(const float4* __restrict__ g, long n4, const float* __restrict__ tail,
                                                    int ntail, float* __restrict__ out) {
  __shared__ float red[32];
  float s[1] = {0.f};
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const float4 v = __ldg(g + i);
    s[0] += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  if (blockIdx.x == 0 && threadIdx.x < ntail) s[0] += tail[threadIdx.x] * tail[threadIdx.x];
  fd_block_sum<1>(s, red);
  if (threadIdx.x == 0) atomicAdd(out, s[0]);
}

// EMA = true also folds the weight EMA into the same pass: the freshly updated parameter is still in a register, so the
// update costs the 8 bytes of reading and writing `ema` and no launch.  torch.lerp's two-branch form, so w = 1 copies.
template <bool EMA>
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                   float* __restrict__ v, float* __restrict__ ema, long n, float lr, float b1,
                                                   float b2, float eps, float wd, float bc1, float bc2_sqrt,
                                                   const float* __restrict__ sumsq, float max_norm, float grad_scale,
                                                   float ema_w) {
  float clip = grad_scale;
  if (sumsq != nullptr && max_norm > 0.f) {
    const float norm = sqrtf(*sumsq) * grad_scale;
    const float c = max_norm / (norm + 1e-6f);
    if (c < 1.f) clip *= c;
  }
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const float pi = p[i];
    const float gi = g[i] * clip + wd * pi;
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float pn = pi - (lr / bc1) * mi / (sqrtf(vi) / bc2_sqrt + eps);
    p[i] = pn;
    if constexpr (EMA) {
      const float e = ema[i];
      ema[i] = ema_w >= 0.5f ? pn - (pn - e) * (1.f - ema_w) : e + ema_w * (pn - e);
    }
  }
}

}  // namespace

extern "C" {

int fd_gn_silu_bwd(const void* h, const void* da, const double* gn_stats, const float* gamma, const float* beta,
                   const float* scale_shift, long ss_stride, void* dh, float* dgamma, float* dbeta, float* dscale_shift,
                   float* dbias, float* workspace, int N, int HW, int C, float eps, void* stream) {
  FD_REQUIRE(h && da && gn_stats && gamma && beta && dh && dgamma && dbeta && workspace && N > 0 && HW > 0,
             "gn_silu_bwd: bad argument");
  FD_REQUIRE(C % 64 == 0 && C <= 1024, "gn_silu_bwd: C=%d must be a multiple of 64, <= 1024", C);
  FD_REQUIRE(scale_shift != nullptr || dscale_shift == nullptr, "gn_silu_bwd: dscale_shift without scale_shift");
  cudaStream_t st = (cudaStream_t)stream;
  const int chunks = C / 8;
  const int ppb = 256 / chunks > 0 ? 256 / chunks : 1;
  const long cap = (long)FD_NUM_SMS * 8 / N + 1;
  long bx = ((long)HW + ppb * 4 - 1) / (ppb * 4);
  if (bx > cap) bx = cap;
  float* coef = workspace;                       // [N][8][2]
  float* partial = workspace + (size_t)N * 16;   // [N][bx][C][3]
  const __nv_bfloat16* hp = static_cast<const __nv_bfloat16*>(h);
  const __nv_bfloat16* dp = static_cast<const __nv_bfloat16*>(da);
  gn_bwd_reduce_kernel<<<dim3((unsigned)bx, (unsigned)N), ppb * chunks, (size_t)ppb * C * 3 * sizeof(float), st>>>(
      hp, dp, gn_stats, gamma, beta, scale_shift, ss_stride, partial, (long)HW, C, eps);
  FD_LAUNCH_CHECK();
  const int cpg = C / 8, slices = 1024 / cpg < 32 ? 1024 / cpg : 32;
  gn_bwd_finalize_kernel<<<dim3((unsigned)N, 8), dim3((unsigned)cpg, (unsigned)slices), 0, st>>>(
      partial, (int)bx, gn_stats, gamma, beta, scale_shift, ss_stride, dgamma, dbeta, dscale_shift, dbias, coef, (long)HW, C, eps);
  FD_LAUNCH_CHECK();
  long bx2 = ((long)HW + ppb * 4 - 1) / (ppb * 4);
  const long cap2 = (long)FD_NUM_SMS * 16 / N + 1;
  if (bx2 > cap2) bx2 = cap2;
  gn_bwd_apply_kernel<<<dim3((unsigned)bx2, (unsigned)N), ppb * chunks, 0, st>>>(
      hp, dp, gn_stats, gamma, beta, scale_shift, ss_stride, coef, static_cast<__nv_bfloat16*>(dh), (long)HW, C, eps);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

size_t fd_gn_silu_bwd_workspace_floats(int N, int C) {
  // coefficients [N][8][2] + per-block partial sums [N][<= 8 * SMs / N + 1 blocks][C][3]
  return (size_t)N * 16 + ((size_t)FD_NUM_SMS * 8 + N) * C * 3;
}

int fd_chan_layernorm_bwd(const void* x, const float* g, const void* dy, const void* add, void* dx, float* dg, long npix,
                          int C, float eps, void* stream) {
  FD_REQUIRE(x && g && dy && dx && dg && npix > 0, "chan_layernorm_bwd: bad argument");
  const __nv_bfloat16* xp = static_cast<const __nv_bfloat16*>(x);
  const __nv_bfloat16* dyp = static_cast<const __nv_bfloat16*>(dy);
  const __nv_bfloat16* ap = static_cast<const __nv_bfloat16*>(add);
  __nv_bfloat16* dxp = static_cast<__nv_bfloat16*>(dx);
  cudaStream_t st = (cudaStream_t)stream;
  switch (C) {
    case 64: chan_ln_bwd_kernel<8, 1><<<egrid(npix * 8, 256, 8), 256, 0, st>>>(xp, g, dyp, ap, dxp, dg, npix, eps); break;
    case 128: chan_ln_bwd_kernel<16, 1><<<egrid(npix * 16, 256, 8), 256, 0, st>>>(xp, g, dyp, ap, dxp, dg, npix, eps); break;
    case 256: chan_ln_bwd_kernel<32, 1><<<egrid(npix * 32, 256, 8), 256, 0, st>>>(xp, g, dyp, ap, dxp, dg, npix, eps); break;
    case 512: chan_ln_bwd_kernel<32, 2><<<egrid(npix * 32, 256, 8), 256, 0, st>>>(xp, g, dyp, ap, dxp, dg, npix, eps); break;
    default: FD_REQUIRE(false, "chan_layernorm_bwd: C=%d not in {64,128,256,512}", C);
  }
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_upsample2x_bwd(const void* dy, void* dx, int N, int H, int W, int C, void* stream) {
  FD_REQUIRE(dy && dx && N > 0 && H > 0 && W > 0 && C % 8 == 0, "upsample2x_bwd: bad argument");
  const long total = (long)N * H * W * (C / 8);
  upsample2x_bwd_kernel<<<egrid(total, 256), 256, 0, (cudaStream_t)stream>>>(static_cast<const uint4*>(dy),
                                                                            static_cast<uint4*>(dx), N, H, W, C / 8);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_add_bf16(const void* a, const void* b, void* out, long n, void* stream) {
  FD_REQUIRE(a && b && out && n > 0 && n % 8 == 0, "add_bf16: bad argument");
  add_bf16_kernel<<<egrid(n / 8, 256), 256, 0, (cudaStream_t)stream>>>(static_cast<const uint4*>(a), static_cast<const uint4*>(b),
                                                                      static_cast<uint4*>(out), n / 8);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_bias_grad(const void* dy, float* db, long npix, int C, void* stream) {
  FD_REQUIRE(dy && db && npix > 0 && C % 8 == 0 && C <= 2048, "bias_grad: bad argument");
  const int chunks = C / 8;
  const int ppb = 256 / chunks > 0 ? 256 / chunks : 1;
  long bx = (npix + ppb * 8 - 1) / (ppb * 8);
  if (bx > FD_NUM_SMS * 8) bx = FD_NUM_SMS * 8;
  bias_grad_kernel<<<(unsigned)bx, ppb * chunks, C * sizeof(float), (cudaStream_t)stream>>>(
      static_cast<const __nv_bfloat16*>(dy), db, npix, C);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_final_conv_bwd(const void* x, const float* w, const float* dout, void* dx, float* dw, float* db, int N, int HW,
                      int Cin, int Cout, void* stream) {
  FD_REQUIRE(x && w && dout && dx && dw && db && N > 0 && HW > 0 && Cout >= 1 && Cout <= 4, "final_conv_bwd: bad argument");
  FD_REQUIRE(Cin == 64, "final_conv_bwd: the UNet's final conv has 64 input channels (got %d)", Cin);
  final_conv_bwd_kernel<<<egrid((long)N * HW * 8, 256, 8), 256, 0, (cudaStream_t)stream>>>(
      static_cast<const __nv_bfloat16*>(x), w, dout, static_cast<__nv_bfloat16*>(dx), dw, db, N, (long)HW, Cout);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_prep_weight_dgrad(const void* wpacked, void* wd, int Cout, int Cin, int taps, void* stream) {
  FD_REQUIRE(wpacked && wd && Cout > 0 && Cin > 0 && taps > 0 && taps <= 65535, "prep_weight_dgrad: bad argument");
  dim3 grid((Cin + 31) / 32, (Cout + 31) / 32, taps);
  prep_weight_dgrad_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(static_cast<const __nv_bfloat16*>(wpacked),
                                                                  static_cast<__nv_bfloat16*>(wd), Cout, Cin, taps);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_prep_weight_bwd(const float* g, const float* w, float* dw, int Cout, int Cin, int KH, int KW, int kind,
                       int standardize, float eps, void* stream) {
  FD_REQUIRE(g && w && dw && Cout > 0 && Cin > 0 && KH > 0 && KW > 0, "prep_weight_bwd: bad argument");
  FD_REQUIRE(kind >= 0 && kind <= 3, "prep_weight_bwd: kind %d", kind);
  FD_REQUIRE(kind != 3 || Cin <= 64, "prep_weight_bwd: kind 3 needs Cin <= 64");
  FD_REQUIRE(kind != 1 || (Cin % 4 == 0 && KH == 1 && KW == 1), "prep_weight_bwd: kind 1 is a 1x1 over 4*C channels");
  FD_REQUIRE(kind != 2 || KW * Cin <= 64, "prep_weight_bwd: kind 2 needs KW*Cin <= 64");
  const int Kp = kind == 2 ? KH * 64 : (kind == 3 ? KH * KW * 64 : Cin * KH * KW);
  prep_weight_bwd_kernel<<<Cout, 256, 0, (cudaStream_t)stream>>>(g, w, dw, Cout, Cin, KH, KW, kind, standardize, eps, Kp);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_prep_weight_dgrad_batch(const long long* table, const int* blk_start, int n_layers, int total_blocks, void* stream) {
  FD_REQUIRE(table && blk_start && n_layers > 0 && total_blocks > 0, "prep_weight_dgrad_batch: bad argument");
  prep_weight_dgrad_batch_kernel<<<total_blocks, 256, 0, (cudaStream_t)stream>>>(table, blk_start, n_layers);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_prep_weight_bwd_batch(const long long* table, const int* blk_start, int n_layers, int total_blocks, float eps,
                             void* stream) {
  FD_REQUIRE(table && blk_start && n_layers > 0 && total_blocks > 0, "prep_weight_bwd_batch: bad argument");
  prep_weight_bwd_batch_kernel<<<total_blocks, 256, 0, (cudaStream_t)stream>>>(table, blk_start, n_layers, eps);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_linear_bwd_w(const float* dY, long dy_stride, const float* X, long x_stride, float* dW, float* db, int B, int J,
                    int K, int act, void* stream) {
  FD_REQUIRE(dY && X && dW && B > 0 && J > 0 && K > 0 && act >= 0 && act <= 2, "linear_bwd_w: bad argument");
  const long total = (long)J * K;
  lin_bwd_w_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(dY, dy_stride, X, x_stride, dW, db, B,
                                                                                     J, K, act);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_linear_bwd_x(const float* dY, long dy_stride, const float* W, const float* A, long a_stride, float* dX,
                    long dx_stride, int B, int J, int K, int act, void* stream) {
  FD_REQUIRE(dY && W && dX && B > 0 && J > 0 && K > 0 && act >= 0 && act <= 2, "linear_bwd_x: bad argument");
  FD_REQUIRE(act == 0 || A != nullptr, "linear_bwd_x: activation needs its forward input");
  FD_REQUIRE(B <= 65535, "linear_bwd_x: batch too large");
  lin_bwd_x_kernel<<<dim3((K + 31) / 32, B), 256, 0, (cudaStream_t)stream>>>(dY, dy_stride, W, A ? A : dY, a_stride, dX,
                                                                            dx_stride, B, J, K, act);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_sumsq(const float* g, long n, float* out, void* stream) {
  FD_REQUIRE(g && out && n > 0, "sumsq: bad argument");
  FD_REQUIRE(((uintptr_t)g & 15) == 0, "sumsq: buffer must be 16-byte aligned");
  const long n4 = n / 4;
  sumsq_kernel<<<egrid(n4 > 0 ? n4 : 1, 256, 8), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(g), n4,
                                                                                g + n4 * 4, (int)(n - n4 * 4), out);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long n, float lr, float beta1,
                 float beta2, float eps, float weight_decay, int step, const float* grad_sumsq, float max_norm,
                 float grad_scale, void* stream) {
  FD_REQUIRE(param && grad && exp_avg && exp_avg_sq && n > 0 && step >= 1, "adam_step: bad argument");
  const float bc1 = 1.f - powf(beta1, (float)step);
  const float bc2 = 1.f - powf(beta2, (float)step);
  adam_kernel<false><<<egrid(n, 256, 8), 256, 0, (cudaStream_t)stream>>>(param, grad, exp_avg, exp_avg_sq, nullptr, n, lr,
                                                                        beta1, beta2, eps, weight_decay, bc1, sqrtf(bc2),
                                                                        grad_sumsq, max_norm, grad_scale, 0.f);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_adam_ema_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, float* ema, long n, float lr,
                     float beta1, float beta2, float eps, float weight_decay, int step, const float* grad_sumsq,
                     float max_norm, float grad_scale, float ema_weight, void* stream) {
  FD_REQUIRE(param && grad && exp_avg && exp_avg_sq && ema && n > 0 && step >= 1, "adam_ema_step: bad argument");
  FD_REQUIRE(ema_weight >= 0.f && ema_weight <= 1.f, "adam_ema_step: ema_weight %g outside [0, 1]", (double)ema_weight);
  const float bc1 = 1.f - powf(beta1, (float)step);
  const float bc2 = 1.f - powf(beta2, (float)step);
  adam_kernel<true><<<egrid(n, 256, 8), 256, 0, (cudaStream_t)stream>>>(param, grad, exp_avg, exp_avg_sq, ema, n, lr, beta1,
                                                                       beta2, eps, weight_decay, bc1, sqrtf(bc2), grad_sumsq,
                                                                       max_norm, grad_scale, ema_weight);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

}  // extern "C"
