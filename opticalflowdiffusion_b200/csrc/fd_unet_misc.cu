// HBM-bound pieces of the UNet forward (denoising_diffusion.py:81-417) on bf16 NHWC activations:
// input packing for the 7x7 init conv, weight standardisation + packing, GroupNorm apply (+ scale /
// shift + SiLU + residual), channel LayerNorm, nearest upsample, time embedding MLPs, final 1x1
// conv, layout conversions.  Every activation kernel moves 16 bytes (8 channels) per access and
// keeps per-channel coefficients in registers across its pixel loop.
#include "fd_common.cuh"

namespace {

int egrid(long items, int threads, int per_sm = 16) {
  long blocks = (items + threads - 1) / threads;
  const long cap = (long)FD_NUM_SMS * per_sm;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

// ---------------------------------------------------------------------------------------------
// Unet.forward input assembly (:367-368) + UnetWithWarp NaN mask (flow_diffuser.py:39-45), emitted
// as the horizontally unrolled tensor the 7x7 init conv consumes as a 7x1 conv over 64 channels:
//   packed[b,h,w, kx*Ctot + c] = in[b,c,h,w+kx-3]   (zero outside the row, zero above 7*Ctot)
// ---------------------------------------------------------------------------------------------
constexpr int kPackPx = 256;       // pixels of one image row per block

__global__ void __launch_bounds__(256) pack_input_kernel(const float* __restrict__ x, const float* __restrict__ cond,
                                                         __nv_bfloat16* __restrict__ packed, int B, int Cx, int Cc,
                                                         int H, int W, int nan_mask, int segs, int H0, int W0, int pt,
                                                         int pl) {
  // x / cond are H0 x W0 planes placed at (pt, pl) inside the H x W frame the UNet runs on; the border is
  // replicate-padded on the fly (InputPadder(mode='sintel') semantics, future/raft_utils.py:7-25): H0 = H, pt = 0 -> none
  // A block owns kPackPx consecutive pixels of one row: the <= 9 input planes (+3 halo pixels per side) are read
  // once, coalesced, into shared memory; then lane q of every 8-lane group writes the q-th 16-byte granule of its
  // pixel, so a warp store covers 4 pixels x 128 B of contiguous memory.
  __shared__ float s_in[9][kPackPx + 6];
  const int Ctot = Cx + (nan_mask ? 1 : 0) + Cc;
  const int seg = blockIdx.x % segs;
  const long row = blockIdx.x / segs;              // b * H + h
  const int b = (int)(row / H), h = (int)(row % H);
  const int w0 = seg * kPackPx;
  const long HW = (long)H0 * W0;
  const int t = threadIdx.x;
  const int hs = min(max(h - pt, 0), H0 - 1);
  for (int idx = t; idx < Ctot * (kPackPx + 6); idx += 256) {
    const int c = idx / (kPackPx + 6), i = idx - c * (kPackPx + 6);
    const int w = w0 + i - 3;
    float v = 0.f;
    if (w >= 0 && w < W) {
      const long p = (long)hs * W0 + min(max(w - pl, 0), W0 - 1);
      if (c < Cx) {
        v = __ldg(x + ((long)b * Cx + c) * HW + p);
      } else if (nan_mask && c == Cx) {
        v = 0.f;                                  // filled below
      } else {
        v = __ldg(cond + ((long)b * Cc + (c - Cx - (nan_mask ? 1 : 0))) * HW + p);
      }
    }
    s_in[c][i] = v;
  }
  __syncthreads();
  if (nan_mask) {       // UnetWithWarp (flow_diffuser.py:39-45): NaN -> 0, mask channel = any NaN over the x channels
    for (int i = t; i < kPackPx + 6; i += 256) {
      bool any_nan = false;
      for (int c = 0; c < Cx; ++c) {
        const float v = s_in[c][i];
        if (v != v) { any_nan = true; s_in[c][i] = 0.f; }
      }
      s_in[Cx][i] = any_nan ? 1.f : 0.f;
    }
    __syncthreads();
  }
  // this thread's granule q = t % 8 is the same for all its pixels: resolve (tap, channel) of its 8 values once
  const int q = t & 7;
  int off[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int k = q * 8 + j;
    const int kx = k / Ctot, c = k - kx * Ctot;
    off[j] = kx < 7 ? c * (kPackPx + 6) + kx : -1;     // s_in[c][px + kx]  (px + kx - 3 + 3)
  }
  const float* sflat = &s_in[0][0];
  uint4* dst = reinterpret_cast<uint4*>(packed + (row * W + w0) * 64);
#pragma unroll 4
  for (int it = 0; it < kPackPx / 32; ++it) {
    const int px = it * 32 + (t >> 3);
    if (w0 + px >= W) break;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = off[j] >= 0 ? sflat[off[j] + px] : 0.f;
    uint4 o;
    o.x = fd_pack_bf16(v[0], v[1]);
    o.y = fd_pack_bf16(v[2], v[3]);
    o.z = fd_pack_bf16(v[4], v[5]);
    o.w = fd_pack_bf16(v[6], v[7]);
    dst[px * 8 + q] = o;
  }
}

// Wide variant for more than 9 input channels (latent mode: flow_diffuser.py:98-110 builds a Unet over latent_dim + ... = 33-35
// channels, flow_pred.py:31-37 one over latent_dim + 3): plain NHWC with the channels zero-padded to 64; init_conv then runs
// as a 49-tap implicit GEMM (weights in fd_prep_weight's kind-3 layout).  Same NaN / mask / replicate-pad semantics as above.
constexpr int kWidePx = 64;

__global__ void __launch_bounds__(256) pack_input_wide_kernel(const float* __restrict__ x, const float* __restrict__ cond,
                                                              __nv_bfloat16* __restrict__ packed, int B, int Cx, int Cc, int H,
                                                              int W, int nan_mask, int segs, int H0, int W0, int pt, int pl) {
  __shared__ float s_in[64][kWidePx + 1];
  const int Ctot = Cx + (nan_mask ? 1 : 0) + Cc;
  const int seg = blockIdx.x % segs;
  const long row = blockIdx.x / segs;              // b * H + h
  const int b = (int)(row / H), h = (int)(row % H);
  const int w0 = seg * kWidePx;
  const long HW = (long)H0 * W0;
  const int t = threadIdx.x;
  const int hs = min(max(h - pt, 0), H0 - 1);
  for (int idx = t; idx < 64 * kWidePx; idx += 256) {
    const int c = idx / kWidePx, i = idx - c * kWidePx;
    const int w = w0 + i;
    float v = 0.f;
    if (c < Ctot && w < W) {
      const long p = (long)hs * W0 + min(max(w - pl, 0), W0 - 1);
      if (c < Cx) v = __ldg(x + ((long)b * Cx + c) * HW + p);
      else if (nan_mask && c == Cx) v = 0.f;
      else v = __ldg(cond + ((long)b * Cc + (c - Cx - (nan_mask ? 1 : 0))) * HW + p);
    }
    s_in[c][i] = v;
  }
  __syncthreads();
  if (nan_mask) {
    for (int i = t; i < kWidePx; i += 256) {
      bool any_nan = false;
      for (int c = 0; c < Cx; ++c) {
        const float v = s_in[c][i];
        if (v != v) { any_nan = true; s_in[c][i] = 0.f; }
      }
      s_in[Cx][i] = any_nan ? 1.f : 0.f;
    }
    __syncthreads();
  }
  const int q = t & 7;
  uint4* dst = reinterpret_cast<uint4*>(packed + (row * W + w0) * 64);
#pragma unroll
  for (int it = 0; it < kWidePx / 32; ++it) {
    const int px = it * 32 + (t >> 3);
    if (w0 + px >= W) break;
    uint4 o;
    o.x = fd_pack_bf16(s_in[q * 8 + 0][px], s_in[q * 8 + 1][px]);
    o.y = fd_pack_bf16(s_in[q * 8 + 2][px], s_in[q * 8 + 3][px]);
    o.z = fd_pack_bf16(s_in[q * 8 + 4][px], s_in[q * 8 + 5][px]);
    o.w = fd_pack_bf16(s_in[q * 8 + 6][px], s_in[q * 8 + 7][px]);
    dst[px * 8 + q] = o;
  }
}

// ---------------------------------------------------------------------------------------------
// weight standardisation (:106-114) + bf16 packing into the implicit-GEMM K order.  One block per
// output channel; statistics in fp32 (biased variance), two passes like the reference's reduce.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void prep_weight_body(const float* __restrict__ w, __nv_bfloat16* __restrict__ packed, int Cin,
                                                 int KH, int KW, int kind, int standardize, float eps, int Kpacked, int o) {
  __shared__ float red[32];
  __shared__ float s_mean, s_rstd;
  const int n = Cin * KH * KW;
  const float* wo = w + (long)o * n;
  float mean = 0.f, rstd = 1.f;
  if (standardize) {
    float s[1] = {0.f};
    for (int i = threadIdx.x; i < n; i += blockDim.x) s[0] += wo[i];
    fd_block_sum<1>(s, red);
    if (threadIdx.x == 0) s_mean = s[0] / (float)n;
    __syncthreads();
    mean = s_mean;
    float v[1] = {0.f};
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const float d = wo[i] - mean;
      v[0] += d * d;
    }
    fd_block_sum<1>(v, red);
    if (threadIdx.x == 0) s_rstd = rsqrtf(v[0] / (float)n + eps);
    __syncthreads();
    rstd = s_rstd;
  }
  __nv_bfloat16* po = packed + (long)o * Kpacked;
  if (kind >= 2) {
    for (int k = threadIdx.x; k < Kpacked; k += blockDim.x) po[k] = __float2bfloat16(0.f);
    __syncthreads();
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    // torch order: i = (ci*KH + ky)*KW + kx
    const int kx = i % KW;
    const int ky = (i / KW) % KH;
    const int ci = i / (KW * KH);
    int k;
    if (kind == 0) {
      k = (ky * KW + kx) * Cin + ci;
    } else if (kind == 1) {
      const int C = Cin / 4;
      k = (ci & 3) * C + (ci >> 2);       // torch channel c*4 + p1*2 + p2 -> (p1*2+p2)*C + c
    } else if (kind == 2) {
      k = ky * 64 + kx * Cin + ci;
    } else {
      k = (ky * KW + kx) * 64 + ci;       // kind 3: tap-major over an input zero-padded to 64 channels (wide init_conv)
    }
    po[k] = __float2bfloat16((wo[i] - mean) * rstd);
  }
}

__global__ void __launch_bounds__(256) prep_weight_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ packed,
                                                          int Cout, int Cin, int KH, int KW, int kind, int standardize,
                                                          float eps, int Kpacked) {
  prep_weight_body(w, packed, Cin, KH, KW, kind, standardize, eps, Kpacked, blockIdx.x);
}

// Upsample (:89-93) = nearest x2 followed by a 3x3 conv.  On the LOW-resolution grid that is four 2x2 convolutions, one per output
// phase (a, b) = (row, column parity): output row 2i + a reads up-sampled rows 2i + a - 1 .. 2i + a + 1, i.e. source rows
// {i-1, i, i} (a = 0) or {i, i, i+1} (a = 1), so the three row taps collapse to two with the weights of the coinciding taps
// ADDED (same for columns).  2.25x fewer MACs than the conv on the up-sampled tensor, which is never materialised.
//   packed[p = a*2+b][co][(ty*2+tx)*Cin + ci] = sum over ky in rows(a, ty), kx in cols(b, tx) of w[co][ci][ky][kx]
//   rows(0,0) = {0}, rows(0,1) = {1,2}, rows(1,0) = {0,1}, rows(1,1) = {2}; tap ty reads source row i + ty - (1 - a).
__global__ void __launch_bounds__(256) prep_weight_upconv_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ packed,
                                                                 int Cout, int Cin) {
  const int co = blockIdx.x, p = blockIdx.y, a = p >> 1, b = p & 1;
  const float* wc = w + (long)co * Cin * 9;
  __nv_bfloat16* dst = packed + ((long)p * Cout + co) * 4 * Cin;
  for (int k = threadIdx.x; k < 4 * Cin; k += 256) {
    const int t = k / Cin, ci = k - t * Cin, ty = t >> 1, tx = t & 1;
    const int ky0 = a == 0 ? (ty == 0 ? 0 : 1) : (ty == 0 ? 0 : 2), ky1 = a == 0 ? (ty == 0 ? 0 : 2) : (ty == 0 ? 1 : 2);
    const int kx0 = b == 0 ? (tx == 0 ? 0 : 1) : (tx == 0 ? 0 : 2), kx1 = b == 0 ? (tx == 0 ? 0 : 2) : (tx == 0 ? 1 : 2);
    float acc = 0.f;
    for (int ky = ky0; ky <= ky1; ++ky)
      for (int kx = kx0; kx <= kx1; ++kx) acc += wc[(ci * 3 + ky) * 3 + kx];
    dst[k] = __float2bfloat16(acc);
  }
}

// all layers in one launch: block -> (layer, output channel) through the prefix sums of the layers' block counts
__global__ void __launch_bounds__(256) prep_weight_batch_kernel(const long long* __restrict__ table,
                                                                const int* __restrict__ blk_start, int n_layers, float eps) {
  int lo = 0, hi = n_layers;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (blk_start[mid] <= (int)blockIdx.x) lo = mid; else hi = mid;
  }
  const long long* r = table + (long)lo * 8;
  const int Cin = (int)r[4], KH = (int)r[5], KW = (int)r[6], kind = (int)(r[7] & 0xff), ws = (int)((r[7] >> 8) & 1);
  const int Kp = kind == 2 ? KH * 64 : (kind == 3 ? KH * KW * 64 : Cin * KH * KW);
  prep_weight_body(reinterpret_cast<const float*>(r[0]), reinterpret_cast<__nv_bfloat16*>(r[1]), Cin, KH, KW, kind, ws, eps, Kp,
                   (int)blockIdx.x - blk_start[lo]);
}

// ---------------------------------------------------------------------------------------------
// GroupNorm(8) apply + (scale+1, shift) + SiLU (+ residual): Block.forward :181-187, ResnetBlock :214
// y = silu(a[c] * x + b[c]) (+ res);  a = rstd*gamma*(scale+1), b = (beta - mean*rstd*gamma)*(scale+1) + shift
// grid = (pixel blocks, N); thread owns one 8-channel chunk for a strided set of pixels.
// ---------------------------------------------------------------------------------------------
// TANH (fd_gn_silu_fast, the inference forward): silu(z) = h + h tanh(h), h = z / 2 -- ONE MUFU op per element (tanh.approx,
// 2^-11 relative, before a bf16 rounding of 2^-9) as in the fused forms of this transform (fd_conv_strip.cu: silu_tanh,
// fd_conv_epi.cuh: epi_silu_half), instead of the ex2 + rcp of fd_silu: at 4 B of traffic per element the two MUFU ops of
// fd_silu were 114 us of pipe time per full-resolution launch against 142 us of DRAM time.  fd_gn_silu (the training forward)
// keeps the exp form: the training step gains nothing from the other one (measured), and its parity tests were pinned on it.
template <bool TANH>
__global__ void __launch_bounds__(256) gn_silu_kernel(const __nv_bfloat16* __restrict__ x, const double* __restrict__ stats,
                                                      const float* __restrict__ gamma, const float* __restrict__ beta,
                                                      const float* __restrict__ scale_shift, long ss_stride,
                                                      const __nv_bfloat16* __restrict__ residual,
                                                      __nv_bfloat16* __restrict__ out, long HW, int C, float eps) {
  const int n = blockIdx.y;
  const int chunks = C >> 3;
  const int chunk = threadIdx.x % chunks;
  const int prow = threadIdx.x / chunks;
  const int ppb = blockDim.x / chunks;     // pixels per block pass
  const int cpg = C >> 3;                  // channels per group (8 groups)
  float a[8], b[8];
  // C % 64 == 0: the thread's 8 channels share one group, so the double-precision mean / rstd are computed once per thread
  // (8 x 3 double divisions / square roots per thread cost ~20 us of every launch)
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
    a[j] = TANH ? 0.5f * ga : ga;            // (exact scaling: the TANH form works on h = z / 2)
    b[j] = TANH ? 0.5f * be : be;
  }
  const long base = (long)n * HW;
  constexpr int U = 4;     // pixels in flight per thread: U independent 16-byte loads before any use
  const long stride = (long)gridDim.x * ppb;
  for (long p0 = (long)blockIdx.x * ppb + prow; p0 < HW; p0 += stride * U) {
    uint4 xv[U], rv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long p = p0 + u * stride;
      if (p < HW) {
        const long off = ((base + p) * C + chunk * 8);
        xv[u] = __ldcs(reinterpret_cast<const uint4*>(x + off));
        if (residual != nullptr) rv[u] = __ldcs(reinterpret_cast<const uint4*>(residual + off));
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long p = p0 + u * stride;
      if (p >= HW) break;
      const long off = ((base + p) * C + chunk * 8);
      const uint32_t xw[4] = {xv[u].x, xv[u].y, xv[u].z, xv[u].w};
      float y[8];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 f = fd_unpack_bf16(xw[e]);
        if (TANH) {
          const float h0 = fmaf(a[2 * e], f.x, b[2 * e]), h1 = fmaf(a[2 * e + 1], f.y, b[2 * e + 1]);
          float t0, t1;
          asm("tanh.approx.f32 %0, %1;" : "=f"(t0) : "f"(h0));
          asm("tanh.approx.f32 %0, %1;" : "=f"(t1) : "f"(h1));
          y[2 * e] = fmaf(h0, t0, h0);
          y[2 * e + 1] = fmaf(h1, t1, h1);
        } else {
          y[2 * e] = fd_silu(a[2 * e] * f.x + b[2 * e]);
          y[2 * e + 1] = fd_silu(a[2 * e + 1] * f.y + b[2 * e + 1]);
        }
      }
      if (residual != nullptr) {
        const uint32_t rw[4] = {rv[u].x, rv[u].y, rv[u].z, rv[u].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 f = fd_unpack_bf16(rw[e]);
          y[2 * e] += f.x;
          y[2 * e + 1] += f.y;
        }
      }
      uint4 o;
      o.x = fd_pack_bf16(y[0], y[1]);
      o.y = fd_pack_bf16(y[2], y[3]);
      o.z = fd_pack_bf16(y[4], y[5]);
      o.w = fd_pack_bf16(y[6], y[7]);
      *reinterpret_cast<uint4*>(out + off) = o;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// channel LayerNorm (:116-125): per pixel over C, biased variance, gain only (+ residual).
// LANES = min(C/8, 32) lanes cooperate on one pixel, each holding C/8/LANES 8-channel chunks.
// ---------------------------------------------------------------------------------------------
template <int LANES, int CHUNKS>
__global__ void __launch_bounds__(256) chan_ln_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ g,
                                                      const __nv_bfloat16* __restrict__ residual,
                                                      __nv_bfloat16* __restrict__ out, long npix, float eps) {
  constexpr int C = LANES * CHUNKS * 8;
  const int sub = threadIdx.x % LANES;
  const long gid = ((long)blockIdx.x * blockDim.x + threadIdx.x) / LANES;
  const long gstride = ((long)gridDim.x * blockDim.x) / LANES;
  float gain[CHUNKS][8];
#pragma unroll
  for (int k = 0; k < CHUNKS; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) gain[k][j] = __ldg(g + (k * LANES + sub) * 8 + j);
  // all lanes of a warp iterate together (shuffles below), out-of-range pixel groups are masked
  const long iters = (npix + gstride - 1) / gstride;
  for (long it = 0; it < iters; ++it) {
    const long p = gid + it * gstride;
    const bool valid = p < npix;
    float v[CHUNKS][8];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < CHUNKS; ++k) {
      uint4 xv = make_uint4(0, 0, 0, 0);
      if (valid) xv = __ldg(reinterpret_cast<const uint4*>(x + p * C + (k * LANES + sub) * 8));
      const uint32_t xw[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 f = fd_unpack_bf16(xw[e]);
        v[k][2 * e] = f.x;
        v[k][2 * e + 1] = f.y;
        s += f.x + f.y;
      }
    }
#pragma unroll
    for (int o = LANES / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s * (1.f / C);
    float ss = 0.f;
#pragma unroll
    for (int k = 0; k < CHUNKS; ++k)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float d = v[k][j] - mean;
        ss += d * d;
      }
#pragma unroll
    for (int o = LANES / 2; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const float rstd = rsqrtf(ss * (1.f / C) + eps);
    if (valid) {
#pragma unroll
      for (int k = 0; k < CHUNKS; ++k) {
        const long off = p * C + (k * LANES + sub) * 8;
        float y[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = (v[k][j] - mean) * rstd * gain[k][j];
        if (residual != nullptr) {
          const uint4 rv = __ldg(reinterpret_cast<const uint4*>(residual + off));
          const uint32_t rw[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 f = fd_unpack_bf16(rw[e]);
            y[2 * e] += f.x;
            y[2 * e + 1] += f.y;
          }
        }
        uint4 o;
        o.x = fd_pack_bf16(y[0], y[1]);
        o.y = fd_pack_bf16(y[2], y[3]);
        o.z = fd_pack_bf16(y[4], y[5]);
        o.w = fd_pack_bf16(y[6], y[7]);
        *reinterpret_cast<uint4*>(out + off) = o;
      }
    }
  }
}

// nearest 2x upsample (:91): (N,H,W,C) -> (N,2H,2W,C), 16-byte granules
__global__ void __launch_bounds__(256) upsample2x_kernel(const uint4* __restrict__ x, uint4* __restrict__ out, long N,
                                                         int H, int W, int C8) {
  const long total = N * H * W * C8;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C8);
    long r = i / C8;
    const int w = (int)(r % W);
    r /= W;
    const int h = (int)(r % H);
    const long n = r / H;
    const uint4 v = __ldg(x + i);
    const long o = ((n * 2 * H + 2 * h) * 2 * W + 2 * w) * C8 + c;
    out[o] = v;
    out[o + C8] = v;
    out[o + (long)2 * W * C8] = v;
    out[o + (long)2 * W * C8 + C8] = v;
  }
}

// SinusoidalPosEmb + Linear + GELU(erf) + Linear (:144-151, 319-324); one block per batch element, one WARP per output
// feature (lanes stride the input features: coalesced weight rows, 8 loads per lane).  The first version gave every thread a
// whole weight row -- 256 dependent, uncoalesced loads -- and took 50 us at the head of every DDIM step.
__global__ void __launch_bounds__(1024) time_embed_kernel(const int64_t* __restrict__ t, const float* __restrict__ w1,
                                                          const float* __restrict__ b1, const float* __restrict__ w2,
                                                          const float* __restrict__ b2, float* __restrict__ temb,
                                                          float* __restrict__ pe_out, float* __restrict__ pre_out, int dim,
                                                          int time_dim) {
  extern __shared__ float sm[];
  float* pe = sm;             // [dim]
  float* hid = sm + dim;      // [time_dim]
  const int b = blockIdx.x;
  const int half = dim / 2;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const float tv = (float)t[b];
  const float lg = logf(10000.f) / (float)(half - 1);
  for (int i = threadIdx.x; i < half; i += blockDim.x) {
    const float f = expf((float)i * -lg);
    const float arg = tv * f;
    pe[i] = sinf(arg);
    pe[half + i] = cosf(arg);
    if (pe_out != nullptr) {
      pe_out[(long)b * dim + i] = pe[i];
      pe_out[(long)b * dim + half + i] = pe[half + i];
    }
  }
  __syncthreads();
  for (int j = warp; j < time_dim; j += nwarps) {
    float acc = 0.f;
    for (int k = lane; k < dim; k += 32) acc += pe[k] * __ldg(w1 + (long)j * dim + k);
    acc = fd_warp_sum(acc);
    if (lane == 0) {
      acc += b1[j];
      hid[j] = 0.5f * acc * (1.f + erff(acc * 0.70710678118654752440f));
      if (pre_out != nullptr) pre_out[(long)b * time_dim + j] = acc;
    }
  }
  __syncthreads();
  for (int j = warp; j < time_dim; j += nwarps) {
    float acc = 0.f;
    for (int k = lane; k < time_dim; k += 32) acc += hid[k] * __ldg(w2 + (long)j * time_dim + k);
    acc = fd_warp_sum(acc);
    if (lane == 0) temb[(long)b * time_dim + j] = acc + b2[j];
  }
}

// ResnetBlock.mlp (:193-196,206) for all blocks at once: out[b][j] = bias[j] + sum_k silu(temb[b][k]) w[j][k]
// one warp per (b, j)
__global__ void __launch_bounds__(256) time_proj_kernel(const float* __restrict__ temb, const float* __restrict__ w,
                                                        const float* __restrict__ bias, float* __restrict__ out, int B,
                                                        int time_dim, int J) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= B * J) return;
  const int b = warp / J, j = warp % J;
  float acc = 0.f;
  for (int k = lane; k < time_dim; k += 32) acc += fd_silu(temb[(long)b * time_dim + k]) * __ldg(w + (long)j * time_dim + k);
  acc = fd_warp_sum(acc);
  if (lane == 0) out[(long)b * J + j] = acc + bias[j];
}

// final 1x1 conv (:361,417): bf16 NHWC (Cin) -> fp32 NCHW (Cout <= 4).  4 lanes share a pixel, each owning a
// contiguous quarter of the channels whose weights it keeps in registers (a warp reads whole 128-byte lines),
// combined with two shuffles.  PER = Cin / 4 (16 for the UNet's 64 channels).
template <int PER>
__global__ void __launch_bounds__(256) final_conv_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w,
                                                         const float* __restrict__ bias, float* __restrict__ out, int N,
                                                         long HW, int CoutAll, int W, int H0, int W0, int pt, int pl,
                                                         int o_base) {
  // output channels o_base .. o_base + 3 of CoutAll (the host loops over groups of four: the flow UNet has 2, the latent
  // autoencoder's encoder 16)
  const int Cout = min(CoutAll - o_base, 4);
  w += (long)o_base * (PER * 4);
  bias += o_base;
  // the H0 x W0 window at (pt, pl) of the H x W frame is written (crop of the internal padding); W0 = W, pt = pl = 0 -> all
  constexpr int Cin = PER * 4;
  const int sub = threadIdx.x & 3;
  float wr[4][PER];
#pragma unroll
  for (int o = 0; o < 4; ++o)
#pragma unroll
    for (int c = 0; c < PER; ++c) wr[o][c] = o < Cout ? __ldg(w + o * Cin + sub * PER + c) : 0.f;
  float br[4];
#pragma unroll
  for (int o = 0; o < 4; ++o) br[o] = o < Cout ? __ldg(bias + o) : 0.f;
  // 32-bit pixel arithmetic (the host checks N * HW < 2^31): the three 64-bit divisions per pixel of the first version cost
  // more instructions than the 64 FMAs
  const unsigned total = (unsigned)((long)N * HW);
  const unsigned gstride = (gridDim.x * blockDim.x) >> 2;
  const unsigned uHW = (unsigned)HW, uW = (unsigned)W;
  const unsigned iters = (total + gstride - 1) / gstride;
  unsigned i = (blockIdx.x * blockDim.x + threadIdx.x) >> 2;
  for (unsigned it = 0; it < iters; ++it, i += gstride) {
    const bool valid = i < total;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    if (valid) {
      const uint4* row = reinterpret_cast<const uint4*>(x + (long)i * Cin + sub * PER);
#pragma unroll
      for (int q = 0; q < PER / 8; ++q) {
        const uint4 xv = __ldg(row + q);
        const uint32_t xw[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 f = fd_unpack_bf16(xw[e]);
#pragma unroll
          for (int o = 0; o < 4; ++o) acc[o] += f.x * wr[o][q * 8 + 2 * e] + f.y * wr[o][q * 8 + 2 * e + 1];
        }
      }
    }
#pragma unroll
    for (int o = 0; o < 4; ++o) {
      acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], 1);
      acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], 2);
    }
    if (valid && sub < Cout) {       // lane `sub` writes output channel `sub`
      const unsigned n = i / uHW, p = i - n * uHW;
      const unsigned hq = p / uW;
      const int hh = (int)hq - pt, ww = (int)(p - hq * uW) - pl;
      const float r = sub == 0 ? acc[0] + br[0] : (sub == 1 ? acc[1] + br[1] : (sub == 2 ? acc[2] + br[2] : acc[3] + br[3]));
      if (hh >= 0 && hh < H0 && ww >= 0 && ww < W0) out[(((long)n * CoutAll + o_base + sub) * H0 + hh) * (long)W0 + ww] = r;
    }
  }
}

__global__ void __launch_bounds__(256) nchw_to_nhwc_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ out,
                                                           int N, int C, long HW) {
  const long total = (long)N * HW * C;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const long r = i / C;
    const long p = r % HW, n = r / HW;
    out[i] = __float2bfloat16(x[(n * C + c) * HW + p]);
  }
}
__global__ void __launch_bounds__(256) nhwc_to_nchw_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ out,
                                                           int N, int C, long HW) {
  const long total = (long)N * HW * C;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long p = i % HW;
    const long r = i / HW;
    const int c = (int)(r % C);
    const long n = r / C;
    out[i] = __bfloat162float(x[(n * HW + p) * C + c]);
  }
}

}  // namespace

extern "C" {

int fd_pack_input_pad(const float* x, const float* cond, void* packed, int B, int Cx, int Cc, int H0, int W0, int pad_top,
                      int pad_left, int H, int W, int nan_mask, void* stream) {
  FD_REQUIRE(x && packed && B > 0 && H0 > 0 && W0 > 0 && Cx > 0 && Cc >= 0, "pack_input_pad: bad argument");
  FD_REQUIRE(cond != nullptr || Cc == 0, "pack_input_pad: Cc > 0 needs cond");
  FD_REQUIRE(pad_top >= 0 && pad_left >= 0 && pad_top + H0 <= H && pad_left + W0 <= W, "pack_input_pad: window outside the frame");
  FD_REQUIRE(Cx + (nan_mask ? 1 : 0) + Cc <= 9, "pack_input_pad: at most 9 input channels (7 taps x 9 <= 64)");
  const int segs = (W + kPackPx - 1) / kPackPx;
  FD_REQUIRE((long)B * H * segs < (1L << 31), "pack_input_pad: too many rows");
  pack_input_kernel<<<(unsigned)((long)B * H * segs), 256, 0, (cudaStream_t)stream>>>(
      x, cond, static_cast<__nv_bfloat16*>(packed), B, Cx, Cc, H, W, nan_mask, segs, H0, W0, pad_top, pad_left);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_pack_input_wide(const float* x, const float* cond, void* packed, int B, int Cx, int Cc, int H0, int W0, int pad_top,
                       int pad_left, int H, int W, int nan_mask, void* stream) {
  FD_REQUIRE(x && packed && B > 0 && H0 > 0 && W0 > 0 && Cx > 0 && Cc >= 0, "pack_input_wide: bad argument");
  FD_REQUIRE(cond != nullptr || Cc == 0, "pack_input_wide: Cc > 0 needs cond");
  FD_REQUIRE(pad_top >= 0 && pad_left >= 0 && pad_top + H0 <= H && pad_left + W0 <= W, "pack_input_wide: window outside the frame");
  FD_REQUIRE(Cx + (nan_mask ? 1 : 0) + Cc <= 64, "pack_input_wide: at most 64 input channels");
  const int segs = (W + kWidePx - 1) / kWidePx;
  FD_REQUIRE((long)B * H * segs < (1L << 31), "pack_input_wide: too many rows");
  pack_input_wide_kernel<<<(unsigned)((long)B * H * segs), 256, 0, (cudaStream_t)stream>>>(
      x, cond, static_cast<__nv_bfloat16*>(packed), B, Cx, Cc, H, W, nan_mask, segs, H0, W0, pad_top, pad_left);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_prep_weight(const float* w, void* packed, int Cout, int Cin, int KH, int KW, int kind, int standardize, float eps,
                   void* stream) {
  FD_REQUIRE(w && packed && Cout > 0 && Cin > 0 && KH > 0 && KW > 0, "prep_weight: bad argument");
  FD_REQUIRE(kind >= 0 && kind <= 3, "prep_weight: kind %d", kind);
  FD_REQUIRE(kind != 3 || Cin <= 64, "prep_weight: kind 3 needs Cin <= 64");
  FD_REQUIRE(kind != 1 || (Cin % 4 == 0 && KH == 1 && KW == 1), "prep_weight: kind 1 is a 1x1 over 4*C channels");
  FD_REQUIRE(kind != 2 || KW * Cin <= 64, "prep_weight: kind 2 needs KW*Cin <= 64");
  const int Kp = kind == 2 ? KH * 64 : (kind == 3 ? KH * KW * 64 : Cin * KH * KW);
  prep_weight_kernel<<<Cout, 256, 0, (cudaStream_t)stream>>>(w, static_cast<__nv_bfloat16*>(packed), Cout, Cin, KH, KW,
                                                             kind, standardize, eps, Kp);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_prep_weight_upconv(const float* w, void* packed, int Cout, int Cin, void* stream) {
  FD_REQUIRE(w && packed && Cout > 0 && Cin > 0, "prep_weight_upconv: bad argument");
  prep_weight_upconv_kernel<<<dim3(Cout, 4), 256, 0, (cudaStream_t)stream>>>(w, static_cast<__nv_bfloat16*>(packed), Cout, Cin);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_prep_weight_batch(const long long* table, const int* blk_start, int n_layers, int total_blocks, float eps, void* stream) {
  FD_REQUIRE(table && blk_start && n_layers > 0 && total_blocks > 0, "prep_weight_batch: bad argument");
  prep_weight_batch_kernel<<<total_blocks, 256, 0, (cudaStream_t)stream>>>(table, blk_start, n_layers, eps);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

static int gn_silu_launch(bool tanh_form, const void* x, const double* gn_stats, const float* gamma, const float* beta,
                          const float* scale_shift, long ss_stride, const void* residual, void* out, int N, int HW, int C,
                          float eps, void* stream) {
  FD_REQUIRE(x && gn_stats && gamma && beta && out && N > 0 && HW > 0, "gn_silu: bad argument");
  FD_REQUIRE(C % 64 == 0 && C <= 2048, "gn_silu: C=%d must be a multiple of 64", C);
  const int chunks = C / 8;
  const int ppb = 256 / chunks > 0 ? 256 / chunks : 1;
  FD_REQUIRE(chunks <= 256, "gn_silu: C too large");
  long bx = ((long)HW + ppb * 4 - 1) / (ppb * 4);
  const long cap = (long)FD_NUM_SMS * 16 / N + 1;
  if (bx > cap) bx = cap;
  dim3 grid((unsigned)bx, (unsigned)N);
  auto kernel = tanh_form ? gn_silu_kernel<true> : gn_silu_kernel<false>;
  kernel<<<grid, ppb * chunks, 0, (cudaStream_t)stream>>>(static_cast<const __nv_bfloat16*>(x), gn_stats, gamma, beta, scale_shift,
                                                          ss_stride, static_cast<const __nv_bfloat16*>(residual),
                                                          static_cast<__nv_bfloat16*>(out), (long)HW, C, eps);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_gn_silu(const void* x, const double* gn_stats, const float* gamma, const float* beta, const float* scale_shift,
               long ss_stride, const void* residual, void* out, int N, int HW, int C, float eps, void* stream) {
  return gn_silu_launch(false, x, gn_stats, gamma, beta, scale_shift, ss_stride, residual, out, N, HW, C, eps, stream);
}

int fd_gn_silu_fast(const void* x, const double* gn_stats, const float* gamma, const float* beta, const float* scale_shift,
                    long ss_stride, const void* residual, void* out, int N, int HW, int C, float eps, void* stream) {
  return gn_silu_launch(true, x, gn_stats, gamma, beta, scale_shift, ss_stride, residual, out, N, HW, C, eps, stream);
}

int fd_chan_layernorm(const void* x, const float* g, const void* residual, void* out, long npix, int C, float eps,
                      void* stream) {
  FD_REQUIRE(x && g && out && npix > 0, "chan_layernorm: bad argument");
  const __nv_bfloat16* xp = static_cast<const __nv_bfloat16*>(x);
  const __nv_bfloat16* rp = static_cast<const __nv_bfloat16*>(residual);
  __nv_bfloat16* op = static_cast<__nv_bfloat16*>(out);
  cudaStream_t st = (cudaStream_t)stream;
  switch (C) {
    case 64: chan_ln_kernel<8, 1><<<egrid(npix * 8, 256), 256, 0, st>>>(xp, g, rp, op, npix, eps); break;
    case 128: chan_ln_kernel<16, 1><<<egrid(npix * 16, 256), 256, 0, st>>>(xp, g, rp, op, npix, eps); break;
    case 256: chan_ln_kernel<32, 1><<<egrid(npix * 32, 256), 256, 0, st>>>(xp, g, rp, op, npix, eps); break;
    case 512: chan_ln_kernel<32, 2><<<egrid(npix * 32, 256), 256, 0, st>>>(xp, g, rp, op, npix, eps); break;
    default: FD_REQUIRE(false, "chan_layernorm: C=%d not in {64,128,256,512}", C);
  }
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_upsample2x(const void* x, void* out, int N, int H, int W, int C, void* stream) {
  FD_REQUIRE(x && out && N > 0 && H > 0 && W > 0 && C % 8 == 0, "upsample2x: bad argument");
  const long total = (long)N * H * W * (C / 8);
  upsample2x_kernel<<<egrid(total, 256), 256, 0, (cudaStream_t)stream>>>(static_cast<const uint4*>(x),
                                                                        static_cast<uint4*>(out), N, H, W, C / 8);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_time_embed(const int64_t* t, const float* w1, const float* b1, const float* w2, const float* b2, float* temb,
                  int B, int dim, int time_dim, void* stream) {
  return fd_time_embed_save(t, w1, b1, w2, b2, temb, nullptr, nullptr, B, dim, time_dim, stream);
}

int fd_time_embed_save(const int64_t* t, const float* w1, const float* b1, const float* w2, const float* b2, float* temb,
                       float* pe, float* pre, int B, int dim, int time_dim, void* stream) {
  FD_REQUIRE(t && w1 && b1 && w2 && b2 && temb && B > 0 && dim >= 4 && dim % 2 == 0 && time_dim > 0, "time_embed: bad argument");
  time_embed_kernel<<<B, 1024, (dim + time_dim) * sizeof(float), (cudaStream_t)stream>>>(t, w1, b1, w2, b2, temb, pe, pre, dim,
                                                                                       time_dim);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_time_proj(const float* temb, const float* w, const float* bias, float* out, int B, int time_dim, int J,
                 void* stream) {
  FD_REQUIRE(temb && w && bias && out && B > 0 && J > 0 && time_dim > 0, "time_proj: bad argument");
  const long threads = (long)B * J * 32;
  time_proj_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(temb, w, bias, out, B, time_dim, J);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_final_conv_crop(const void* x, const float* w, const float* bias, float* out, int N, int H, int W, int Cin, int Cout,
                       int pad_top, int pad_left, int H0, int W0, void* stream) {
  FD_REQUIRE(x && w && bias && out && N > 0 && H > 0 && W > 0 && Cout >= 1 && Cout <= 64, "final_conv_crop: bad argument");
  FD_REQUIRE(Cin == 64, "final_conv_crop: the UNet's final conv has 64 input channels (got %d)", Cin);
  FD_REQUIRE(pad_top >= 0 && pad_left >= 0 && pad_top + H0 <= H && pad_left + W0 <= W && H0 > 0 && W0 > 0,
             "final_conv_crop: window outside the frame");
  FD_REQUIRE((long)N * H * W < (1L << 31), "final_conv_crop: too many pixels");
  for (int o = 0; o < Cout; o += 4) {
    final_conv_kernel<16><<<egrid((long)N * H * W * 4, 256), 256, 0, (cudaStream_t)stream>>>(
        static_cast<const __nv_bfloat16*>(x), w, bias, out, N, (long)H * W, Cout, W, H0, W0, pad_top, pad_left, o);
    FD_LAUNCH_CHECK();
  }
  return FD_OK;
}

int fd_nchw_to_nhwc_bf16(const float* x, void* out, int N, int C, int HW, void* stream) {
  FD_REQUIRE(x && out && N > 0 && C > 0 && HW > 0, "nchw_to_nhwc: bad argument");
  nchw_to_nhwc_kernel<<<egrid((long)N * C * HW, 256), 256, 0, (cudaStream_t)stream>>>(x, static_cast<__nv_bfloat16*>(out), N, C, (long)HW);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_nhwc_bf16_to_nchw(const void* x, float* out, int N, int C, int HW, void* stream) {
  FD_REQUIRE(x && out && N > 0 && C > 0 && HW > 0, "nhwc_to_nchw: bad argument");
  nhwc_to_nchw_kernel<<<egrid((long)N * C * HW, 256), 256, 0, (cudaStream_t)stream>>>(static_cast<const __nv_bfloat16*>(x), out, N, C, (long)HW);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

}  // extern "C"
