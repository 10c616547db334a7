// Backward of the two attention cores (autograd of denoising_diffusion.py:229-243 and :256-267) on
// bf16 NHWC qkv = (N, HW, 384) = [q | k | v], 4 heads x 32.
//
// LinearAttention, with  qs = softmax_d(q) * 32^-0.5,  ks = softmax_pixels(k),  ctx[d,e] = sum_p ks[d,p] v[e,p] / HW,
// out[e,p] = sum_d ctx[d,e] qs[d,p]:
//     dctx[d,e] = sum_p qs[d,p] dout[e,p]                                   (pass 1: reduction over pixels)
//     dqs[d,p]  = sum_e ctx[d,e] dout[e,p] ;   dq = scale * sm (dqs - <sm, dqs>)
//     dv[e,p]   = sum_d ks[d,p] dctx[d,e] / HW
//     dks[d,p]  = sum_e dctx[d,e] v[e,p] / HW ; dk = ks (dks - r[d]),  r[d] = sum_p ks dks = sum_e dctx[d,e] ctx[d,e]
//   so the k softmax over ALL pixels needs no second reduction pass: r comes from the two 32x32 matrices.
//   Pass 2 is one thread per (pixel, head) with the 32x32 matrices broadcast from shared memory.
//
// Attention (flash-style backward, bf16 mma.sync m16n8k16, S / P recomputed from the saved log-sum-exp):
//     D[q] = <dO[q], O[q]> ;  P = exp2(S' - lse) ;  dS = P (dO V^T - D)
//     dQ = scale dS K    (one CTA per 128 queries, streams K/V tiles)
//     dK = scale dS^T Q, dV = P^T dO   (one CTA per 128 keys, streams Q/dO tiles; works on S^T so that the
//     accumulator fragments of P^T / dS^T are directly the A fragments of the two products -- no transposes)
//   No atomics: run-to-run bit-stable.
#include "fd_mma.cuh"

using namespace fdmma;

namespace {

constexpr float kScale = 0.17677669529663687f;          // 32^-0.5
constexpr int kStatsFloats = 2 * kHidden + kHeads * kD * kD;

__device__ __forceinline__ void unpack8(const uint4& v, float* f) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 p = fd_unpack_bf16(w[e]);
    f[2 * e] = p.x;
    f[2 * e + 1] = p.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  uint4 o;
  o.x = fd_pack_bf16(f[0], f[1]);
  o.y = fd_pack_bf16(f[2], f[3]);
  o.z = fd_pack_bf16(f[4], f[5]);
  o.w = fd_pack_bf16(f[6], f[7]);
  return o;
}

// ------------------------------------------------------------------------------------------------
// linear attention backward, pass 1 (tensor cores, K = pixels):
//   dctx[n][head][d][e] += sum over a pixel chunk of qs[p,d] dout[p,e]
// 8 warps = 4 heads x 2 halves of e; 64-pixel tiles of [q(128) | dout(128)] rows, cp.async double buffered.
// A = qs^T via ldmatrix.trans of the raw q rows, softmax over d done in the A-fragment registers (4 values per
// pixel column in a thread, the rest across the 8 lanes that share tq); B = dout via ldmatrix.trans.
// ------------------------------------------------------------------------------------------------
constexpr int kLbTile = 64;
constexpr int kLbRowBytes = 2 * kHidden * 2 + 16;       // 528: conflict-free ldmatrix
constexpr int kLbTileBytes = kLbTile * kLbRowBytes;
constexpr int kLbSmemBytes = 2 * kLbTileBytes;

__global__ void __launch_bounds__(256, 3) linattn_bwd_dctx_kernel(const __nv_bfloat16* __restrict__ qkv,
                                                                  const __nv_bfloat16* __restrict__ dout,
                                                                  float* __restrict__ dctx, int HW, int chunk_px) {
  extern __shared__ __align__(16) uint8_t lb_smem[];
  const int n = blockIdx.y;
  const int p_begin = blockIdx.x * chunk_px;
  const int p_end = min(HW, p_begin + chunk_px);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int g = lane >> 2, tq = lane & 3;
  const int head = warp & 3, nhalf = warp >> 2;
  const __nv_bfloat16* qbase = qkv + (long)n * HW * kQkv;
  const __nv_bfloat16* dbase = dout + (long)n * HW * kHidden;
  const uint32_t smem0 = smem_addr(lb_smem);
  float acc[2][2][4];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[a][b][c] = 0.f;

  auto issue_tile = [&](int p0, int buf) {
    // 64 pixels x 32 granules of 16 B: granules 0..15 = q, 16..31 = dout
#pragma unroll
    for (int it = 0; it < (kLbTile * 32) / 256; ++it) {
      const int idx = it * 256 + t;
      const int px = idx >> 5, q16 = idx & 31;
      const int p = p0 + px;
      const bool ok = p < p_end;
      const long pp = ok ? p : p_begin;
      const __nv_bfloat16* src = q16 < 16 ? qbase + pp * kQkv + q16 * 8 : dbase + pp * kHidden + (q16 - 16) * 8;
      cp_async16(smem0 + buf * kLbTileBytes + px * kLbRowBytes + q16 * 16, src, ok);
    }
    cp_async_commit();
  };
  const int ntiles = (p_end - p_begin + kLbTile - 1) / kLbTile;
  if (ntiles > 0) issue_tile(p_begin, 0);
  const int mi = lane >> 3, r = lane & 7;
  for (int ti = 0; ti < ntiles; ++ti) {
    const int buf = ti & 1;
    const int p0 = p_begin + ti * kLbTile;
    if (ti + 1 < ntiles) {
      issue_tile(p0 + kLbTile, buf ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const uint32_t tb = smem0 + buf * kLbTileBytes;
#pragma unroll
    for (int ks = 0; ks < kLbTile / 16; ++ks) {
      // raw q as A fragments (d x pixel) for both 16-row halves of d
      uint32_t qa[2][4];
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
        ldmatrix_x4_trans(qa[mt], tb + (ks * 16 + (mi >> 1) * 8 + r) * kLbRowBytes + (head * kD + mt * 16 + (mi & 1) * 8) * 2);
      // element (mt, rg, half): d = mt*16 + g (+8 for rg odd), pixel = ks*16 + 2*tq + half (+8 for rg >= 2)
      float v[2][4][2];
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int rg = 0; rg < 4; ++rg) {
          const float2 f = fd_unpack_bf16(qa[mt][rg]);
          v[mt][rg][0] = f.x;
          v[mt][rg][1] = f.y;
        }
#pragma unroll
      for (int ph = 0; ph < 2; ++ph)          // pixel half: rg >> 1
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          float mx = fmaxf(fmaxf(v[0][2 * ph][hf], v[0][2 * ph + 1][hf]), fmaxf(v[1][2 * ph][hf], v[1][2 * ph + 1][hf]));
          mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 4));
          mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 8));
          mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 16));
          float sum = 0.f;
#pragma unroll
          for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int o = 0; o < 2; ++o) {
              const float e = __expf(v[mt][2 * ph + o][hf] - mx);
              v[mt][2 * ph + o][hf] = e;
              sum += e;
            }
          sum += __shfl_xor_sync(0xffffffffu, sum, 4);
          sum += __shfl_xor_sync(0xffffffffu, sum, 8);
          sum += __shfl_xor_sync(0xffffffffu, sum, 16);
          const float inv = kScale / sum;
#pragma unroll
          for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int o = 0; o < 2; ++o) v[mt][2 * ph + o][hf] *= inv;
        }
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int rg = 0; rg < 4; ++rg) qa[mt][rg] = fd_pack_bf16(v[mt][rg][0], v[mt][rg][1]);
      // B (trans): m0 (px 0-7, e 0-7) m1 (px 8-15, e 0-7) m2 (px 0-7, e 8-15) m3 (px 8-15, e 8-15) of this warp's 16 e's
      uint32_t b[4];
      ldmatrix_x4_trans(b, tb + (ks * 16 + (mi & 1) * 8 + r) * kLbRowBytes + (kHidden + head * kD + nhalf * 16 + (mi >> 1) * 8) * 2);
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        mma_bf16(acc[mt][0], qa[mt], b[0], b[1]);
        mma_bf16(acc[mt][1], qa[mt], b[2], b[3]);
      }
    }
    __syncthreads();
  }
  // per-chunk partial (combined in a fixed order by linattn_bwd_dctx_combine_kernel: run-to-run stable, no atomics)
  float* dst = dctx + (((long)n * gridDim.x + blockIdx.x) * kHeads + head) * kD * kD;
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
      const int d = mt * 16 + g, e = nhalf * 16 + nt * 8 + 2 * tq;
      dst[d * kD + e] = acc[mt][nt][0];
      dst[d * kD + e + 1] = acc[mt][nt][1];
      dst[(d + 8) * kD + e] = acc[mt][nt][2];
      dst[(d + 8) * kD + e + 1] = acc[mt][nt][3];
    }
}

__global__ void __launch_bounds__(256) linattn_bwd_dctx_combine_kernel(const float* __restrict__ partial, float* __restrict__ dctx,
                                                                       int N, int chunks) {
  const int per = kHeads * kD * kD;
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long)N * per) return;
  const int n = (int)(i / per), j = (int)(i - (long)n * per);
  float s = 0.f;
  for (int c = 0; c < chunks; ++c) s += partial[((long)n * chunks + c) * per + j];
  dctx[i] = s;
}

// ------------------------------------------------------------------------------------------------
// linear attention backward, pass 2 (tensor cores): per 16-pixel warp tile and head, three 16x32x32 products
//   dqs = dout ctx^T ;  dks = v dctx^T ;  dv = ks dctx
// with the operands loaded straight into accumulator (C) layout from global memory, so that the softmaxes, the
// elementwise backward formulas and the re-packing into A fragments all happen in registers.  ctx / dctx are bf16
// in shared memory ([d][e], rows padded to 80 B).
// ------------------------------------------------------------------------------------------------
constexpr int kMatStride = kD + 8;

// 4x4 transpose of 32-bit words across the 4 lanes of a quad: x[j] of lane i  <->  x[i] of lane j
__device__ __forceinline__ void quad_transpose(uint32_t (&x)[4], int tq) {
  const bool lo1 = (tq & 1) == 0, lo2 = (tq & 2) == 0;
  uint32_t r0 = __shfl_xor_sync(0xffffffffu, lo1 ? x[1] : x[0], 1);
  uint32_t r1 = __shfl_xor_sync(0xffffffffu, lo1 ? x[3] : x[2], 1);
  if (lo1) { x[1] = r0; x[3] = r1; } else { x[0] = r0; x[2] = r1; }
  r0 = __shfl_xor_sync(0xffffffffu, lo2 ? x[2] : x[0], 2);
  r1 = __shfl_xor_sync(0xffffffffu, lo2 ? x[3] : x[1], 2);
  if (lo2) { x[2] = r0; x[3] = r1; } else { x[0] = r0; x[1] = r1; }
}
// 32 channels of two pixel rows into accumulator (C) layout: each lane loads ONE 16-byte granule per row (a quad
// covers the head's 64 contiguous bytes -> full sectors), then the quad transposes so that lane tq holds columns
// nt*8 + 2*tq, +1 of every 8-column tile nt.
__device__ __forceinline__ void load_c(uint32_t (&r)[4][2], const __nv_bfloat16* row0, const __nv_bfloat16* row1, bool ok0,
                                       bool ok1, int tq) {
  uint4 a = make_uint4(0, 0, 0, 0), b = make_uint4(0, 0, 0, 0);
  if (ok0) a = __ldg(reinterpret_cast<const uint4*>(row0 + tq * 8));
  if (ok1) b = __ldg(reinterpret_cast<const uint4*>(row1 + tq * 8));
  uint32_t x[4] = {a.x, a.y, a.z, a.w}, y[4] = {b.x, b.y, b.z, b.w};
  quad_transpose(x, tq);
  quad_transpose(y, tq);
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) {
    r[nt][0] = x[nt];
    r[nt][1] = y[nt];
  }
}
// the inverse: packed C-layout pairs -> one 16-byte store per lane and row
__device__ __forceinline__ void store_c(uint32_t (&x)[4], uint32_t (&y)[4], __nv_bfloat16* row0, __nv_bfloat16* row1, bool ok0,
                                        bool ok1, int tq) {
  quad_transpose(x, tq);
  quad_transpose(y, tq);
  if (ok0) *reinterpret_cast<uint4*>(row0 + tq * 8) = make_uint4(x[0], x[1], x[2], x[3]);
  if (ok1) *reinterpret_cast<uint4*>(row1 + tq * 8) = make_uint4(y[0], y[1], y[2], y[3]);
}
__device__ __forceinline__ void c_to_a(uint32_t (&a)[2][4], const uint32_t (&c)[4][2]) {
#pragma unroll
  for (int kk = 0; kk < 2; ++kk) {
    a[kk][0] = c[2 * kk][0];
    a[kk][1] = c[2 * kk][1];
    a[kk][2] = c[2 * kk + 1][0];
    a[kk][3] = c[2 * kk + 1][1];
  }
}

__global__ void __launch_bounds__(128, 6) linattn_bwd_apply_kernel(const __nv_bfloat16* __restrict__ qkv,
                                                                const __nv_bfloat16* __restrict__ dout,
                                                                const float* __restrict__ stats,
                                                                const float* __restrict__ dctx,
                                                                __nv_bfloat16* __restrict__ dqkv, int HW) {
  __shared__ __align__(16) __nv_bfloat16 s_ctx[kHeads * kD * kMatStride];
  __shared__ __align__(16) __nv_bfloat16 s_dctx[kHeads * kD * kMatStride];
  __shared__ float s_m[kHidden], s_iz[kHidden], s_r[kHidden], s_cmean[kHidden];
  const int n = blockIdx.y;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int g = lane >> 2, tq = lane & 3;
  const float* st = stats + (long)n * kStatsFloats;
  const float* dc = dctx + (long)n * kHeads * kD * kD;
  const float inv_hw = 1.f / (float)HW;
  // ctx[d,e] is the k-softmax average of v_e (/ HW): when v carries an offset common to the pixels, every row d holds about
  // the same value and dq = scale sm (dqs - <sm, dqs>) keeps only the small d-dependent part of dqs = dout ctx^T.  dq is
  // unchanged by a shift of ctx that depends on e only (sum_d sm = 1), so ctx is centred over d before its bf16 rounding:
  // the rounding then scales with that d-dependent part instead of with the offset.
  {
    const float* col = st + 2 * kHidden + (t >> 5) * kD * kD + (t & 31);
    float s = 0.f;
#pragma unroll
    for (int d = 0; d < kD; ++d) s += col[d * kD];
    s_cmean[t] = s * (1.f / kD);
  }
  __syncthreads();
  for (int i = t; i < kHeads * kD * kD; i += 128) {
    const int row = i >> 5, e = i & 31;
    s_ctx[row * kMatStride + e] = __float2bfloat16(st[2 * kHidden + i] - s_cmean[(row >> 5) * kD + e]);
    s_dctx[row * kMatStride + e] = __float2bfloat16(dc[i]);
  }
  s_m[t] = st[t];
  s_iz[t] = 1.f / st[kHidden + t];
  {
    float r = 0.f;      // r[d] = sum_e dctx[d,e] ctx[d,e]   (fp32 sources, ctx not centred)
#pragma unroll
    for (int e = 0; e < kD; ++e) r += dc[t * kD + e] * st[2 * kHidden + t * kD + e];
    s_r[t] = r;
  }
  __syncthreads();
  const uint32_t ctx_s = smem_addr(s_ctx), dctx_s = smem_addr(s_dctx);
  const int mi = lane >> 3, r8 = lane & 7;
  const long nbase = (long)n * HW;
  for (int p0 = (blockIdx.x * 4 + warp) * 16; p0 < HW; p0 += gridDim.x * 64) {
    const int pr0 = p0 + g, pr1 = p0 + g + 8;
    const bool ok0 = pr0 < HW, ok1 = pr1 < HW;
    const __nv_bfloat16* row0 = qkv + (nbase + (ok0 ? pr0 : 0)) * kQkv;
    const __nv_bfloat16* row1 = qkv + (nbase + (ok1 ? pr1 : 0)) * kQkv;
    const __nv_bfloat16* do0 = dout + (nbase + (ok0 ? pr0 : 0)) * kHidden;
    const __nv_bfloat16* do1 = dout + (nbase + (ok1 ? pr1 : 0)) * kHidden;
    __nv_bfloat16* dr0 = dqkv + (nbase + (ok0 ? pr0 : 0)) * kQkv;
    __nv_bfloat16* dr1 = dqkv + (nbase + (ok1 ? pr1 : 0)) * kQkv;
#pragma unroll 1
    for (int head = 0; head < kHeads; ++head) {
      const int hc = head * kD;
      const uint32_t cm = ctx_s + head * kD * kMatStride * 2, dm = dctx_s + head * kD * kMatStride * 2;
      // ---------------- dq
      {
        uint32_t qc[4][2], dc_[4][2], da[2][4];
        load_c(qc, row0 + hc, row1 + hc, ok0, ok1, tq);
        load_c(dc_, do0 + hc, do1 + hc, ok0, ok1, tq);
        c_to_a(da, dc_);
        float sm[4][4], dqs[4][4];
        float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          const float2 a = fd_unpack_bf16(qc[nt][0]), b = fd_unpack_bf16(qc[nt][1]);
          sm[nt][0] = a.x; sm[nt][1] = a.y; sm[nt][2] = b.x; sm[nt][3] = b.y;
          mx0 = fmaxf(mx0, fmaxf(a.x, a.y));
          mx1 = fmaxf(mx1, fmaxf(b.x, b.y));
        }
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
        float s0 = 0.f, s1 = 0.f;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          sm[nt][0] = __expf(sm[nt][0] - mx0); sm[nt][1] = __expf(sm[nt][1] - mx0);
          sm[nt][2] = __expf(sm[nt][2] - mx1); sm[nt][3] = __expf(sm[nt][3] - mx1);
          s0 += sm[nt][0] + sm[nt][1];
          s1 += sm[nt][2] + sm[nt][3];
        }
        s0 += __shfl_xor_sync(0xffffffffu, s0, 1); s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
        s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
        const float i0 = 1.f / s0, i1 = 1.f / s1;
        float dot0 = 0.f, dot1 = 0.f;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {       // n = d tile; B[k = e][n = d] = ctx[d][e]
#pragma unroll
          for (int i = 0; i < 4; ++i) dqs[nt][i] = 0.f;
          uint32_t bf[4];
          ldmatrix_x4(bf, cm + ((nt * 8 + r8) * kMatStride + mi * 8) * 2);
          mma_bf16(dqs[nt], da[0], bf[0], bf[1]);
          mma_bf16(dqs[nt], da[1], bf[2], bf[3]);
          sm[nt][0] *= i0; sm[nt][1] *= i0; sm[nt][2] *= i1; sm[nt][3] *= i1;
          dot0 += sm[nt][0] * dqs[nt][0] + sm[nt][1] * dqs[nt][1];
          dot1 += sm[nt][2] * dqs[nt][2] + sm[nt][3] * dqs[nt][3];
        }
        dot0 += __shfl_xor_sync(0xffffffffu, dot0, 1); dot0 += __shfl_xor_sync(0xffffffffu, dot0, 2);
        dot1 += __shfl_xor_sync(0xffffffffu, dot1, 1); dot1 += __shfl_xor_sync(0xffffffffu, dot1, 2);
        uint32_t o0[4], o1[4];
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          o0[nt] = fd_pack_bf16(kScale * sm[nt][0] * (dqs[nt][0] - dot0), kScale * sm[nt][1] * (dqs[nt][1] - dot0));
          o1[nt] = fd_pack_bf16(kScale * sm[nt][2] * (dqs[nt][2] - dot1), kScale * sm[nt][3] * (dqs[nt][3] - dot1));
        }
        store_c(o0, o1, dr0 + hc, dr1 + hc, ok0, ok1, tq);
      }
      // ---------------- dk, dv
      {
        uint32_t kc[4][2], vc[4][2], va[2][4], ka[2][4];
        load_c(kc, row0 + kHidden + hc, row1 + kHidden + hc, ok0, ok1, tq);
        load_c(vc, row0 + 2 * kHidden + hc, row1 + 2 * kHidden + hc, ok0, ok1, tq);
        c_to_a(va, vc);
        float ks[4][4];
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          const int d = hc + nt * 8 + 2 * tq;
          const float2 a = fd_unpack_bf16(kc[nt][0]), b = fd_unpack_bf16(kc[nt][1]);
          ks[nt][0] = __expf(a.x - s_m[d]) * s_iz[d];
          ks[nt][1] = __expf(a.y - s_m[d + 1]) * s_iz[d + 1];
          ks[nt][2] = __expf(b.x - s_m[d]) * s_iz[d];
          ks[nt][3] = __expf(b.y - s_m[d + 1]) * s_iz[d + 1];
          kc[nt][0] = fd_pack_bf16(ks[nt][0], ks[nt][1]);
          kc[nt][1] = fd_pack_bf16(ks[nt][2], ks[nt][3]);
        }
        c_to_a(ka, kc);
        uint32_t k0[4], k1[4];
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {       // dks[p, d] = sum_e v[p,e] dctx[d,e]
          float dks[4] = {0.f, 0.f, 0.f, 0.f};
          uint32_t bf[4];
          ldmatrix_x4(bf, dm + ((nt * 8 + r8) * kMatStride + mi * 8) * 2);
          mma_bf16(dks, va[0], bf[0], bf[1]);
          mma_bf16(dks, va[1], bf[2], bf[3]);
          const int d = hc + nt * 8 + 2 * tq;
          const float r0 = s_r[d], r1 = s_r[d + 1];
          k0[nt] = fd_pack_bf16(ks[nt][0] * (dks[0] * inv_hw - r0), ks[nt][1] * (dks[1] * inv_hw - r1));
          k1[nt] = fd_pack_bf16(ks[nt][2] * (dks[2] * inv_hw - r0), ks[nt][3] * (dks[3] * inv_hw - r1));
        }
        store_c(k0, k1, dr0 + kHidden + hc, dr1 + kHidden + hc, ok0, ok1, tq);
        float dv[4][4];
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
          for (int i = 0; i < 4; ++i) dv[nt][i] = 0.f;
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {       // dv[p, e] = sum_d ks[p,d] dctx[d,e] : B[k = d][n = e] row-major -> trans
          uint32_t b01[4], b23[4];
          const uint32_t ba = dm + ((kk * 16 + (mi & 1) * 8 + r8) * kMatStride + (mi >> 1) * 8) * 2;
          ldmatrix_x4_trans(b01, ba);
          ldmatrix_x4_trans(b23, ba + 16 * 2);
          mma_bf16(dv[0], ka[kk], b01[0], b01[1]);
          mma_bf16(dv[1], ka[kk], b01[2], b01[3]);
          mma_bf16(dv[2], ka[kk], b23[0], b23[1]);
          mma_bf16(dv[3], ka[kk], b23[2], b23[3]);
        }
        uint32_t v0[4], v1[4];
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          v0[nt] = fd_pack_bf16(dv[nt][0] * inv_hw, dv[nt][1] * inv_hw);
          v1[nt] = fd_pack_bf16(dv[nt][2] * inv_hw, dv[nt][3] * inv_hw);
        }
        store_c(v0, v1, dr0 + 2 * kHidden + hc, dr1 + 2 * kHidden + hc, ok0, ok1, tq);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// full attention backward
// ------------------------------------------------------------------------------------------------
constexpr int kRowStride = kD + 8;                 // bf16 per staged row: 80 B, conflict-free ldmatrix
constexpr int kTile = 64;                          // streamed rows per tile
constexpr int kTileElems = kTile * kRowStride;

// D[n][head][p] = sum_d dO[p][head*32+d] * O[p][head*32+d]
__global__ void __launch_bounds__(256) attn_bwd_prep_kernel(const __nv_bfloat16* __restrict__ o,
                                                            const __nv_bfloat16* __restrict__ dout, float* __restrict__ D,
                                                            int N, int HW) {
  const long total = (long)N * HW * kHeads;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int head = (int)(i % kHeads);
    const long np = i / kHeads;
    const long n = np / HW, p = np - n * HW;
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float a[8], b[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(o + np * kHidden + head * kD + j * 8)), a);
      unpack8(__ldg(reinterpret_cast<const uint4*>(dout + np * kHidden + head * kD + j * 8)), b);
#pragma unroll
      for (int e = 0; e < 8; ++e) s += a[e] * b[e];
    }
    D[(n * kHeads + head) * HW + p] = s;
  }
}

// A fragments (16 rows x 32 d) of rows row0 = base + g, row1 = row0 + 8 straight from global memory
__device__ __forceinline__ void load_a_frags(uint32_t (&a)[2][4], const __nv_bfloat16* base, long row_stride, int row0,
                                             int row1, int HW, int col0, int tq) {
#pragma unroll
  for (int kk = 0; kk < 2; ++kk) {
    const int c0 = col0 + kk * 16 + 2 * tq;
    a[kk][0] = row0 < HW ? __ldg(reinterpret_cast<const uint32_t*>(base + (long)row0 * row_stride + c0)) : 0u;
    a[kk][1] = row1 < HW ? __ldg(reinterpret_cast<const uint32_t*>(base + (long)row1 * row_stride + c0)) : 0u;
    a[kk][2] = row0 < HW ? __ldg(reinterpret_cast<const uint32_t*>(base + (long)row0 * row_stride + c0 + 8)) : 0u;
    a[kk][3] = row1 < HW ? __ldg(reinterpret_cast<const uint32_t*>(base + (long)row1 * row_stride + c0 + 8)) : 0u;
  }
}

// dQ: CTA = 128 queries (8 warps x 16), streams K / V tiles of 64 keys
__global__ void __launch_bounds__(256) attn_bwd_dq_kernel(const __nv_bfloat16* __restrict__ qkv,
                                                          const __nv_bfloat16* __restrict__ dout,
                                                          const float* __restrict__ lse, const float* __restrict__ Dv,
                                                          __nv_bfloat16* __restrict__ dqkv, int HW, float scale_log2) {
  __shared__ __align__(16) __nv_bfloat16 s_k[2][kTileElems];
  __shared__ __align__(16) __nv_bfloat16 s_v[2][kTileElems];
  const int n = blockIdx.z, head = blockIdx.y;
  const int q0 = blockIdx.x * 128;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int g = lane >> 2, tq = lane & 3;
  const __nv_bfloat16* base = qkv + (long)n * HW * kQkv;
  const __nv_bfloat16* dbase = dout + (long)n * HW * kHidden;
  const int row0 = q0 + warp * 16 + g, row1 = row0 + 8;
  uint32_t qa[2][4], da[2][4];
  load_a_frags(qa, base, kQkv, row0, row1, HW, head * kD, tq);
  load_a_frags(da, dbase, kHidden, row0, row1, HW, head * kD, tq);
  const long sb = ((long)n * kHeads + head) * HW;
  const float lse0 = row0 < HW ? lse[sb + row0] : 0.f, lse1 = row1 < HW ? lse[sb + row1] : 0.f;
  const float D0 = row0 < HW ? Dv[sb + row0] : 0.f, D1 = row1 < HW ? Dv[sb + row1] : 0.f;
  float acc[4][4];
#pragma unroll
  for (int dt = 0; dt < 4; ++dt)
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[dt][i] = 0.f;

  const uint32_t sk = smem_addr(&s_k[0][0]), sv = smem_addr(&s_v[0][0]);
  auto issue_tile = [&](int k0, int buf) {
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int idx = it * 256 + t;
      const int key = (idx >> 2) & 63, part = idx & 3, is_v = idx >> 8;
      const int kg = k0 + key;
      const bool ok = kg < HW;
      const __nv_bfloat16* src = base + (long)(ok ? kg : 0) * kQkv + (1 + is_v) * kHidden + head * kD + part * 8;
      cp_async16((is_v ? sv : sk) + (buf * kTileElems + key * kRowStride + part * 8) * 2, src, ok);
    }
    cp_async_commit();
  };
  const int ntiles = (HW + kTile - 1) / kTile;
  issue_tile(0, 0);
  const int mi = lane >> 3, r8 = lane & 7;
  for (int ti = 0; ti < ntiles; ++ti) {
    const int buf = ti & 1, k0 = ti * kTile;
    cp_async_wait<0>();
    __syncthreads();
    if (ti + 1 < ntiles) issue_tile(k0 + kTile, buf ^ 1);
    const uint32_t kb = sk + buf * kTileElems * 2, vb = sv + buf * kTileElems * 2;
    float s[8][4], dp[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
      for (int i = 0; i < 4; ++i) s[nt][i] = dp[nt][i] = 0.f;
      uint32_t kf[4], vf[4];
      ldmatrix_x4(kf, kb + ((nt * 8 + r8) * kRowStride + mi * 8) * 2);
      ldmatrix_x4(vf, vb + ((nt * 8 + r8) * kRowStride + mi * 8) * 2);
      mma_bf16(s[nt], qa[0], kf[0], kf[1]);
      mma_bf16(s[nt], qa[1], kf[2], kf[3]);
      mma_bf16(dp[nt], da[0], vf[0], vf[1]);
      mma_bf16(dp[nt], da[1], vf[2], vf[3]);
    }
    const bool tail = k0 + kTile > HW;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const bool ok = !tail || (k0 + nt * 8 + 2 * tq + (i & 1)) < HW;
        const float p = ok ? exp2f(s[nt][i] * scale_log2 - (i < 2 ? lse0 : lse1)) : 0.f;
        s[nt][i] = p * (dp[nt][i] - (i < 2 ? D0 : D1));      // dS
      }
    }
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      uint32_t pa[4];
      pa[0] = fd_pack_bf16(s[2 * kk][0], s[2 * kk][1]);
      pa[1] = fd_pack_bf16(s[2 * kk][2], s[2 * kk][3]);
      pa[2] = fd_pack_bf16(s[2 * kk + 1][0], s[2 * kk + 1][1]);
      pa[3] = fd_pack_bf16(s[2 * kk + 1][2], s[2 * kk + 1][3]);
      uint32_t k01[4], k23[4];
      const uint32_t ka = kb + ((kk * 16 + (mi & 1) * 8 + r8) * kRowStride + (mi >> 1) * 8) * 2;
      ldmatrix_x4_trans(k01, ka);
      ldmatrix_x4_trans(k23, ka + 16 * 2);
      mma_bf16(acc[0], pa, k01[0], k01[1]);
      mma_bf16(acc[1], pa, k01[2], k01[3]);
      mma_bf16(acc[2], pa, k23[0], k23[1]);
      mma_bf16(acc[3], pa, k23[2], k23[3]);
    }
  }
  __nv_bfloat16* ob = dqkv + (long)n * HW * kQkv + head * kD;
#pragma unroll
  for (int dt = 0; dt < 4; ++dt) {
    if (row0 < HW)
      *reinterpret_cast<uint32_t*>(ob + (long)row0 * kQkv + dt * 8 + 2 * tq) = fd_pack_bf16(acc[dt][0] * kScale, acc[dt][1] * kScale);
    if (row1 < HW)
      *reinterpret_cast<uint32_t*>(ob + (long)row1 * kQkv + dt * 8 + 2 * tq) = fd_pack_bf16(acc[dt][2] * kScale, acc[dt][3] * kScale);
  }
}

// dK, dV: CTA = 128 keys (8 warps x 16), streams Q / dO tiles of 64 queries (+ their lse / D)
__global__ void __launch_bounds__(256) attn_bwd_dkv_kernel(const __nv_bfloat16* __restrict__ qkv,
                                                           const __nv_bfloat16* __restrict__ dout,
                                                           const float* __restrict__ lse, const float* __restrict__ Dv,
                                                           __nv_bfloat16* __restrict__ dqkv, int HW, float scale_log2) {
  __shared__ __align__(16) __nv_bfloat16 s_q[2][kTileElems];
  __shared__ __align__(16) __nv_bfloat16 s_do[2][kTileElems];
  __shared__ float s_lse[2][kTile], s_D[2][kTile];
  const int n = blockIdx.z, head = blockIdx.y;
  const int key0 = blockIdx.x * 128;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int g = lane >> 2, tq = lane & 3;
  const __nv_bfloat16* base = qkv + (long)n * HW * kQkv;
  const __nv_bfloat16* dbase = dout + (long)n * HW * kHidden;
  const int row0 = key0 + warp * 16 + g, row1 = row0 + 8;
  uint32_t ka[2][4], va[2][4];
  load_a_frags(ka, base, kQkv, row0, row1, HW, kHidden + head * kD, tq);
  load_a_frags(va, base, kQkv, row0, row1, HW, 2 * kHidden + head * kD, tq);
  const long sb = ((long)n * kHeads + head) * HW;
  float dk[4][4], dv[4][4];
#pragma unroll
  for (int dt = 0; dt < 4; ++dt)
#pragma unroll
    for (int i = 0; i < 4; ++i) dk[dt][i] = dv[dt][i] = 0.f;

  const uint32_t sq = smem_addr(&s_q[0][0]), sd = smem_addr(&s_do[0][0]);
  auto issue_tile = [&](int q0, int buf) {
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int idx = it * 256 + t;
      const int r = (idx >> 2) & 63, part = idx & 3, is_do = idx >> 8;
      const int qg = q0 + r;
      const bool ok = qg < HW;
      const __nv_bfloat16* src = is_do ? dbase + (long)(ok ? qg : 0) * kHidden + head * kD + part * 8
                                       : base + (long)(ok ? qg : 0) * kQkv + head * kD + part * 8;
      cp_async16((is_do ? sd : sq) + (buf * kTileElems + r * kRowStride + part * 8) * 2, src, ok);
    }
    cp_async_commit();
    if (t < kTile) {
      const int qg = q0 + t;
      s_lse[buf][t] = qg < HW ? lse[sb + qg] : INFINITY;      // P = exp2(. - inf) = 0 for rows past the end
      s_D[buf][t] = qg < HW ? Dv[sb + qg] : 0.f;
    }
  };
  const int ntiles = (HW + kTile - 1) / kTile;
  issue_tile(0, 0);
  const int mi = lane >> 3, r8 = lane & 7;
  for (int ti = 0; ti < ntiles; ++ti) {
    const int buf = ti & 1, q0 = ti * kTile;
    cp_async_wait<0>();
    __syncthreads();
    if (ti + 1 < ntiles) issue_tile(q0 + kTile, buf ^ 1);
    const uint32_t qb = sq + buf * kTileElems * 2, db = sd + buf * kTileElems * 2;
    // S^T (16 keys x 64 queries) and dP^T = V dO^T
    float s[8][4], dp[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
      for (int i = 0; i < 4; ++i) s[nt][i] = dp[nt][i] = 0.f;
      uint32_t qf[4], df[4];
      ldmatrix_x4(qf, qb + ((nt * 8 + r8) * kRowStride + mi * 8) * 2);
      ldmatrix_x4(df, db + ((nt * 8 + r8) * kRowStride + mi * 8) * 2);
      mma_bf16(s[nt], ka[0], qf[0], qf[1]);
      mma_bf16(s[nt], ka[1], qf[2], qf[3]);
      mma_bf16(dp[nt], va[0], df[0], df[1]);
      mma_bf16(dp[nt], va[1], df[2], df[3]);
    }
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const int qc = nt * 8 + 2 * tq;
      const float l0 = s_lse[buf][qc], l1 = s_lse[buf][qc + 1];
      const float d0 = s_D[buf][qc], d1 = s_D[buf][qc + 1];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float p = exp2f(s[nt][i] * scale_log2 - ((i & 1) ? l1 : l0));
        s[nt][i] = p;                                           // P^T
        dp[nt][i] = p * (dp[nt][i] - ((i & 1) ? d1 : d0));      // dS^T
      }
    }
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      uint32_t pa[4], sa[4];
      pa[0] = fd_pack_bf16(s[2 * kk][0], s[2 * kk][1]);
      pa[1] = fd_pack_bf16(s[2 * kk][2], s[2 * kk][3]);
      pa[2] = fd_pack_bf16(s[2 * kk + 1][0], s[2 * kk + 1][1]);
      pa[3] = fd_pack_bf16(s[2 * kk + 1][2], s[2 * kk + 1][3]);
      sa[0] = fd_pack_bf16(dp[2 * kk][0], dp[2 * kk][1]);
      sa[1] = fd_pack_bf16(dp[2 * kk][2], dp[2 * kk][3]);
      sa[2] = fd_pack_bf16(dp[2 * kk + 1][0], dp[2 * kk + 1][1]);
      sa[3] = fd_pack_bf16(dp[2 * kk + 1][2], dp[2 * kk + 1][3]);
      uint32_t b01[4], b23[4];
      const uint32_t off = ((kk * 16 + (mi & 1) * 8 + r8) * kRowStride + (mi >> 1) * 8) * 2;
      ldmatrix_x4_trans(b01, db + off);         // dO[k = query][n = d]
      ldmatrix_x4_trans(b23, db + off + 16 * 2);
      mma_bf16(dv[0], pa, b01[0], b01[1]);
      mma_bf16(dv[1], pa, b01[2], b01[3]);
      mma_bf16(dv[2], pa, b23[0], b23[1]);
      mma_bf16(dv[3], pa, b23[2], b23[3]);
      ldmatrix_x4_trans(b01, qb + off);         // Q[k = query][n = d]
      ldmatrix_x4_trans(b23, qb + off + 16 * 2);
      mma_bf16(dk[0], sa, b01[0], b01[1]);
      mma_bf16(dk[1], sa, b01[2], b01[3]);
      mma_bf16(dk[2], sa, b23[0], b23[1]);
      mma_bf16(dk[3], sa, b23[2], b23[3]);
    }
  }
  __nv_bfloat16* ob = dqkv + (long)n * HW * kQkv + head * kD;
#pragma unroll
  for (int dt = 0; dt < 4; ++dt) {
    const int c = dt * 8 + 2 * tq;
    if (row0 < HW) {
      *reinterpret_cast<uint32_t*>(ob + (long)row0 * kQkv + kHidden + c) = fd_pack_bf16(dk[dt][0] * kScale, dk[dt][1] * kScale);
      *reinterpret_cast<uint32_t*>(ob + (long)row0 * kQkv + 2 * kHidden + c) = fd_pack_bf16(dv[dt][0], dv[dt][1]);
    }
    if (row1 < HW) {
      *reinterpret_cast<uint32_t*>(ob + (long)row1 * kQkv + kHidden + c) = fd_pack_bf16(dk[dt][2] * kScale, dk[dt][3] * kScale);
      *reinterpret_cast<uint32_t*>(ob + (long)row1 * kQkv + 2 * kHidden + c) = fd_pack_bf16(dv[dt][2], dv[dt][3]);
    }
  }
}

}  // namespace

extern "C" {

size_t fd_linattn_stats_floats(void) { return kStatsFloats; }

static int lb_chunks(int N, int HW, int* chunk_px) {
  int want = (FD_NUM_SMS * 3) / N;
  if (want < 1) want = 1;
  int px = (HW + want - 1) / want;
  px = ((px + kLbTile - 1) / kLbTile) * kLbTile;
  *chunk_px = px;
  return (HW + px - 1) / px;
}

size_t fd_linattn_bwd_workspace_floats(int N, int HW) {
  int px;
  const int chunks = lb_chunks(N, HW, &px);
  return (size_t)N * kStatsFloats + (size_t)N * (chunks + 1) * kHeads * kD * kD + fd_linattn_workspace_floats(N, HW);
}

int fd_linattn_bwd(const void* qkv, const void* dout, void* dqkv, const float* saved_stats, float* workspace, int N, int HW,
                   void* stream) {
  FD_REQUIRE(qkv && dout && dqkv && workspace && N > 0 && HW > 0, "linattn_bwd: bad argument");
  FD_REQUIRE(N <= 65535, "linattn_bwd: batch too large");
  cudaStream_t st = (cudaStream_t)stream;
  int px;
  const int chunks = lb_chunks(N, HW, &px);
  float* stats = workspace;
  float* dctx = stats + (size_t)N * kStatsFloats;
  float* dpart = dctx + (size_t)N * kHeads * kD * kD;                 // [N][chunks][4][32][32]
  float* fwd_ws = dpart + (size_t)N * chunks * kHeads * kD * kD;
  const __nv_bfloat16* q = static_cast<const __nv_bfloat16*>(qkv);
  const __nv_bfloat16* dO = static_cast<const __nv_bfloat16*>(dout);
  if (saved_stats != nullptr) {
    stats = const_cast<float*>(saved_stats);      // from fd_linattn_save: no recomputation of the k softmax statistics
  } else if (int e = fd_linattn_stats(q + kHidden, kQkv, stats, fwd_ws, N, HW, stream)) {
    return e;
  }
  static bool attr_set = false;
  if (!attr_set) {
    FD_CUDA(cudaFuncSetAttribute(linattn_bwd_dctx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLbSmemBytes));
    attr_set = true;
  }
  linattn_bwd_dctx_kernel<<<dim3(chunks, N), 256, kLbSmemBytes, st>>>(q, dO, dpart, HW, px);
  FD_LAUNCH_CHECK();
  linattn_bwd_dctx_combine_kernel<<<(N * kHeads * kD * kD + 255) / 256, 256, 0, st>>>(dpart, dctx, N, chunks);
  FD_LAUNCH_CHECK();
  int bx = (HW + 63) / 64;
  const int cap = (FD_NUM_SMS * 8 + N - 1) / N;
  if (bx > cap) bx = cap;
  linattn_bwd_apply_kernel<<<dim3(bx, N), 128, 0, st>>>(q, dO, stats, dctx, static_cast<__nv_bfloat16*>(dqkv), HW);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

size_t fd_attention_bwd_workspace_floats(int N, int HW) { return (size_t)N * kHeads * HW; }

int fd_attention_bwd(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, float* workspace,
                     int N, int HW, void* stream) {
  FD_REQUIRE(qkv && out && dout && lse && dqkv && workspace && N > 0 && HW > 0, "attention_bwd: bad argument");
  FD_REQUIRE(N <= 65535, "attention_bwd: batch too large");
  cudaStream_t st = (cudaStream_t)stream;
  const float scale_log2 = kScale * 1.4426950408889634f;
  const __nv_bfloat16* q = static_cast<const __nv_bfloat16*>(qkv);
  const __nv_bfloat16* dO = static_cast<const __nv_bfloat16*>(dout);
  float* D = workspace;
  long blocks = ((long)N * HW * kHeads + 255) / 256;
  if (blocks > FD_NUM_SMS * 16) blocks = FD_NUM_SMS * 16;
  attn_bwd_prep_kernel<<<(unsigned)blocks, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(out), dO, D, N, HW);
  FD_LAUNCH_CHECK();
  const dim3 grid((HW + 127) / 128, kHeads, N);
  attn_bwd_dq_kernel<<<grid, 256, 0, st>>>(q, dO, lse, D, static_cast<__nv_bfloat16*>(dqkv), HW, scale_log2);
  FD_LAUNCH_CHECK();
  attn_bwd_dkv_kernel<<<grid, 256, 0, st>>>(q, dO, lse, D, static_cast<__nv_bfloat16*>(dqkv), HW, scale_log2);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

}  // extern "C"
