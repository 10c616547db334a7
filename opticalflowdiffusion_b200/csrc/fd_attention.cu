// Attention cores of the UNet on bf16 NHWC qkv = (N, HW, 384) = [q | k | v], 4 heads x 32.
//
// LinearAttention (denoising_diffusion.py:229-243): softmax(q) over d, softmax(k) over ALL pixels,
//   ctx[d,e] = sum_n k[d,n] v[e,n] / HW,  out[e,n] = sum_d ctx[d,e] q[d,n] * 32^-0.5.
//   O(HW) and bandwidth-bound: three launches
//     (1) per pixel-chunk partial (running max, sum of exp, 32x32 context) with online rescaling,
//     (2) combine chunks -> ctx (N,4,32,32) fp32,
//     (3) apply: per pixel softmax_d(q) and the 32x32 product, ctx broadcast from shared memory.
// Attention (:256-267): fd_attention / fd_attention_lse launch the tcgen05 kernel of fd_attention_tc.cu.

#include "fd_mma.cuh"

using namespace fdmma;

namespace {


// ------------------------------------------------------------------------------------------------
// linear attention, pass 1: per pixel-chunk partial (running max m, sum of exp s, 32x32 context per head)
//   ctx[d,e] = sum_n exp(k[d,n] - m[d]) v[e,n]  as a tensor-core GEMM with K = pixels:
//   A[d][n] = exp(k) and B[n][e] = v both live in smem as [pixel][channel] rows -> ldmatrix.trans.
//   8 warps = 4 heads x 2 halves of d; cp.async double-buffered 64-pixel tiles.
// ------------------------------------------------------------------------------------------------
constexpr int kLaTile = 64;                                   // pixels per smem tile
constexpr int kLaRowBytes = 2 * kHidden * 2 + 16;             // k|v bf16 row + 16 B pad (conflict-free ldmatrix)
constexpr int kLaTileBytes = kLaTile * kLaRowBytes;
constexpr int kLaSmemBytes = 2 * kLaTileBytes;
constexpr int kLaPartial = 2 * kHidden + kHeads * kD * kD;    // m[128], s[128], ctx[4][32][32]

__global__ void __launch_bounds__(256, 3) linattn_partial_kernel(const __nv_bfloat16* __restrict__ kv, int row_stride,
                                                              float* __restrict__ partial, int HW, int chunk_px) {
  extern __shared__ __align__(16) uint8_t la_smem[];
  const int n = blockIdx.y, chunk = blockIdx.x;
  const int p_begin = chunk * chunk_px;
  const int p_end = min(HW, p_begin + chunk_px);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int g = lane >> 2, tq = lane & 3;
  const int head = warp & 3, mhalf = warp >> 2;      // this warp owns ctx rows d = mhalf*16 + {g, g+8} of `head`
  const __nv_bfloat16* base = kv + (long)n * HW * row_stride;        // rows of [k(128) | v(128)], row_stride elements apart
  const uint32_t smem0 = smem_addr(la_smem);
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  // running max / sum of exp of the two k channels (rows) this thread sees; the 4 lanes of a quad hold the same max
  // and disjoint partial sums
  float m0 = -INFINITY, m1 = -INFINITY, s0 = 0.f, s1 = 0.f;

  auto issue_tile = [&](int p0, int buf) {
    // 64 pixels x 32 granules of 16 B (k|v = 512 B per pixel): 8 cp.async per thread
#pragma unroll
    for (int it = 0; it < (kLaTile * 32) / 256; ++it) {
      const int idx = it * 256 + t;
      const int px = idx >> 5, q16 = idx & 31;
      const int p = p0 + px;
      const bool ok = p < p_end;
      cp_async16(smem0 + buf * kLaTileBytes + px * kLaRowBytes + q16 * 16, base + (long)(ok ? p : p_begin) * row_stride + q16 * 8, ok);
    }
    cp_async_commit();
  };

  const int ntiles = (p_end - p_begin + kLaTile - 1) / kLaTile;
  if (ntiles > 0) issue_tile(p_begin, 0);
  const int mi = lane >> 3, r = lane & 7;       // ldmatrix: lanes 8*mi..8*mi+7 address matrix mi, row r
  for (int ti = 0; ti < ntiles; ++ti) {
    const int buf = ti & 1;
    const int p0 = p_begin + ti * kLaTile;
    if (ti + 1 < ntiles) {
      issue_tile(p0 + kLaTile, buf ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const uint32_t tb = smem0 + buf * kLaTileBytes;
    const int nvalid = p_end - p0;                 // >= 64 except in the chunk's last tile
    // ---- raw k as A fragments (d x pixel): m0 (px 0-7, d 0-7), m1 (px 0-7, d 8-15), m2 (px 8-15, d 0-7), m3 (px 8-15, d 8-15)
    uint32_t ka[kLaTile / 16][4];
#pragma unroll
    for (int ks = 0; ks < kLaTile / 16; ++ks)
      ldmatrix_x4_trans(ka[ks], tb + (ks * 16 + (mi >> 1) * 8 + r) * kLaRowBytes + (head * kD + mhalf * 16 + (mi & 1) * 8) * 2);
    // element (ks, reg, half): row d = g (+8 for reg 1,3), pixel = ks*16 + 2*tq + half (+8 for reg 2,3)
    float t0 = -INFINITY, t1 = -INFINITY;
#pragma unroll
    for (int ks = 0; ks < kLaTile / 16; ++ks) {
#pragma unroll
      for (int rg = 0; rg < 4; ++rg) {
        const float2 f = fd_unpack_bf16(ka[ks][rg]);
        const int px = ks * 16 + 2 * tq + (rg >> 1) * 8;
        const float a = px < nvalid ? f.x : -INFINITY, b = px + 1 < nvalid ? f.y : -INFINITY;
        if (rg & 1) t1 = fmaxf(t1, fmaxf(a, b)); else t0 = fmaxf(t0, fmaxf(a, b));
      }
    }
    t0 = fmaxf(t0, __shfl_xor_sync(0xffffffffu, t0, 1)); t0 = fmaxf(t0, __shfl_xor_sync(0xffffffffu, t0, 2));
    t1 = fmaxf(t1, __shfl_xor_sync(0xffffffffu, t1, 1)); t1 = fmaxf(t1, __shfl_xor_sync(0xffffffffu, t1, 2));
    const float mn0 = fmaxf(m0, t0), mn1 = fmaxf(m1, t1);
    const float f0 = (m0 == -INFINITY) ? 0.f : __expf(m0 - mn0), f1 = (m1 == -INFINITY) ? 0.f : __expf(m1 - mn1);
    m0 = mn0;
    m1 = mn1;
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      acc[nt][0] *= f0; acc[nt][1] *= f0; acc[nt][2] *= f1; acc[nt][3] *= f1;
    }
    float e0 = 0.f, e1 = 0.f;
#pragma unroll
    for (int ks = 0; ks < kLaTile / 16; ++ks) {
#pragma unroll
      for (int rg = 0; rg < 4; ++rg) {
        const float2 f = fd_unpack_bf16(ka[ks][rg]);
        const int px = ks * 16 + 2 * tq + (rg >> 1) * 8;
        const float mm = (rg & 1) ? mn1 : mn0;
        const float a = px < nvalid ? __expf(f.x - mm) : 0.f, b = px + 1 < nvalid ? __expf(f.y - mm) : 0.f;
        const uint32_t pk = fd_pack_bf16(a, b);
        ka[ks][rg] = pk;
        const float2 rq = fd_unpack_bf16(pk);     // the normaliser sums exactly what the GEMM consumes
        if (rg & 1) e1 += rq.x + rq.y; else e0 += rq.x + rq.y;
      }
    }
    s0 = s0 * f0 + e0;
    s1 = s1 * f1 + e1;
    // ---- ctx += exp(k) v^T : K = 64 pixels, N = 32 e
#pragma unroll
    for (int ks = 0; ks < kLaTile / 16; ++ks) {
      uint32_t b01[4], b23[4];
      // B (trans): m0 (px 0-7, e 0-7) m1 (px 8-15, e 0-7) m2 (px 0-7, e 8-15) m3 (px 8-15, e 8-15)
      const uint32_t vb = tb + (ks * 16 + (mi & 1) * 8 + r) * kLaRowBytes + (kHidden + head * kD + (mi >> 1) * 8) * 2;
      ldmatrix_x4_trans(b01, vb);
      ldmatrix_x4_trans(b23, vb + 16 * 2);
      mma_bf16(acc[0], ka[ks], b01[0], b01[1]);
      mma_bf16(acc[1], ka[ks], b01[2], b01[3]);
      mma_bf16(acc[2], ka[ks], b23[0], b23[1]);
      mma_bf16(acc[3], ka[ks], b23[2], b23[3]);
    }
    __syncthreads();     // this buffer is refilled by the prefetch of the next iteration
  }
  s0 += __shfl_xor_sync(0xffffffffu, s0, 1); s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
  s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
  float* out = partial + ((long)n * gridDim.x + chunk) * kLaPartial;
  if (tq == 0) {
    const int d0 = head * kD + mhalf * 16 + g;
    out[d0] = m0;
    out[d0 + 8] = m1;
    out[kHidden + d0] = s0;
    out[kHidden + d0 + 8] = s1;
  }
  float* c = out + 2 * kHidden + (head * kD + mhalf * 16) * kD;
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) {
    c[g * kD + nt * 8 + 2 * tq] = acc[nt][0];
    c[g * kD + nt * 8 + 2 * tq + 1] = acc[nt][1];
    c[(g + 8) * kD + nt * 8 + 2 * tq] = acc[nt][2];
    c[(g + 8) * kD + nt * 8 + 2 * tq + 1] = acc[nt][3];
  }
}

// pass 2: one block per (n, head), thread = (d, e); emits ctx^T in bf16 ([e][d]) for the apply GEMM
__global__ void __launch_bounds__(1024) linattn_combine_kernel(const float* __restrict__ partial,
                                                               __nv_bfloat16* __restrict__ ctx_t, int nchunks,
                                                               float inv_hw) {
  const int n = blockIdx.x / kHeads, head = blockIdx.x % kHeads;
  const int d = threadIdx.x >> 5, e = threadIdx.x & 31;
  const float* base = partial + (long)n * nchunks * kLaPartial;
  float M = -INFINITY;
  for (int c = 0; c < nchunks; ++c) M = fmaxf(M, base[(long)c * kLaPartial + head * kD + d]);
  float S = 0.f, acc = 0.f;
  for (int c = 0; c < nchunks; ++c) {
    const float* pc = base + (long)c * kLaPartial;
    const float mc = pc[head * kD + d];
    const float f = (mc == -INFINITY) ? 0.f : __expf(mc - M);
    S += pc[kHidden + head * kD + d] * f;
    acc += pc[2 * kHidden + (head * kD + d) * kD + e] * f;
  }
  // 32^-0.5 (the q scale, :238) is folded in here so the apply pass only normalises its softmax
  ctx_t[((long)n * kHeads + head) * kD * kD + e * kD + d] = __float2bfloat16(acc / S * inv_hw * 0.17677669529663687f);
}

// pass 2 for the backward pass: fp32 statistics per sample: m[128] (max over pixels of k), Z[128] (sum of exp(k - m)),
// ctx[4][32 d][32 e] = softmax_n(k) v^T / HW (without the q scale)
__global__ void __launch_bounds__(1024) linattn_combine_stats_kernel(const float* __restrict__ partial,
                                                                     float* __restrict__ stats, int nchunks, float inv_hw) {
  const int n = blockIdx.x / kHeads, head = blockIdx.x % kHeads;
  const int d = threadIdx.x >> 5, e = threadIdx.x & 31;
  const float* base = partial + (long)n * nchunks * kLaPartial;
  float M = -INFINITY;
  for (int c = 0; c < nchunks; ++c) M = fmaxf(M, base[(long)c * kLaPartial + head * kD + d]);
  float S = 0.f, acc = 0.f;
  for (int c = 0; c < nchunks; ++c) {
    const float* pc = base + (long)c * kLaPartial;
    const float mc = pc[head * kD + d];
    const float f = (mc == -INFINITY) ? 0.f : __expf(mc - M);
    S += pc[kHidden + head * kD + d] * f;
    acc += pc[2 * kHidden + (head * kD + d) * kD + e] * f;
  }
  float* so = stats + (long)n * kLaPartial;
  if (e == 0) {
    so[head * kD + d] = M;
    so[kHidden + head * kD + d] = S;
  }
  so[2 * kHidden + (head * kD + d) * kD + e] = acc / S * inv_hw;
}

// pass 3: out[n, e] = sum_d softmax_d(q[n, :])[d] ctx[d, e] on tensor cores.
//   block = 4 warps, tile = 64 pixels; warp = 16 pixels x 4 heads; q tile staged by cp.async, A fragments by
//   ldmatrix, softmax in registers (4 lanes share a row), result staged in the warp's own smem rows and
//   written back as 16-byte coalesced stores.
constexpr int kApRowBytes = kHidden * 2 + 16;
constexpr int kCtStride = kD + 8;                   // bf16 per ctx^T row (conflict-free 32-bit fragment loads)

__global__ void __launch_bounds__(128) linattn_apply_kernel(const __nv_bfloat16* __restrict__ qkv,
                                                            const __nv_bfloat16* __restrict__ ctx_t,
                                                            __nv_bfloat16* __restrict__ out, int HW) {
  __shared__ __align__(16) uint8_t s_q[64 * kApRowBytes];
  __shared__ __align__(16) __nv_bfloat16 s_ct[kHeads * kD * kCtStride];
  const int n = blockIdx.y;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int g = lane >> 2, tq = lane & 3;
  for (int i = t; i < kHeads * kD * kD; i += 128) {
    const int hd = i / kD, d = i % kD;               // hd = head*32 + e
    s_ct[hd * kCtStride + d] = ctx_t[(long)n * kHeads * kD * kD + i];
  }
  const __nv_bfloat16* base = qkv + (long)n * HW * kQkv;
  const uint32_t sq = smem_addr(s_q);
  const int ntiles = (HW + 63) / 64;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int p0 = tile * 64;
    __syncthreads();       // previous tile fully written out (and s_ct ready on the first pass)
#pragma unroll
    for (int it = 0; it < (64 * 16) / 128; ++it) {
      const int idx = it * 128 + t;
      const int px = idx >> 4, q16 = idx & 15;
      const bool ok = p0 + px < HW;
      cp_async16(sq + px * kApRowBytes + q16 * 16, base + (long)(ok ? p0 + px : p0) * kQkv + q16 * 8, ok);
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    const uint32_t wrow = sq + (warp * 16) * kApRowBytes;
    const int mi = lane >> 3, r = lane & 7;
    uint32_t qa[kHeads][2][4];
#pragma unroll
    for (int h = 0; h < kHeads; ++h)
#pragma unroll
      for (int ks = 0; ks < 2; ++ks)   // m0 (px 0-7, d 0-7) m1 (px 8-15, d 0-7) m2 (px 0-7, d 8-15) m3 (px 8-15, d 8-15)
        ldmatrix_x4(qa[h][ks], wrow + ((mi & 1) * 8 + r) * kApRowBytes + (h * kD + ks * 16 + (mi >> 1) * 8) * 2);
    __syncwarp();          // all q fragments are in registers: the warp's rows can now receive the output
#pragma unroll
    for (int h = 0; h < kHeads; ++h) {
      float q0[8], q1[8];  // row g / row g+8: d = ks*16 + {2t, 2t+1, 2t+8, 2t+9}
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {
        const float2 a0 = fd_unpack_bf16(qa[h][ks][0]), a1 = fd_unpack_bf16(qa[h][ks][1]);
        const float2 a2 = fd_unpack_bf16(qa[h][ks][2]), a3 = fd_unpack_bf16(qa[h][ks][3]);
        q0[ks * 4 + 0] = a0.x; q0[ks * 4 + 1] = a0.y; q0[ks * 4 + 2] = a2.x; q0[ks * 4 + 3] = a2.y;
        q1[ks * 4 + 0] = a1.x; q1[ks * 4 + 1] = a1.y; q1[ks * 4 + 2] = a3.x; q1[ks * 4 + 3] = a3.y;
      }
      float m0 = q0[0], m1 = q1[0];
#pragma unroll
      for (int i = 1; i < 8; ++i) { m0 = fmaxf(m0, q0[i]); m1 = fmaxf(m1, q1[i]); }
      m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
      m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
      m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
      m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
      float s0 = 0.f, s1 = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        q0[i] = __expf(q0[i] - m0); s0 += q0[i];
        q1[i] = __expf(q1[i] - m1); s1 += q1[i];
      }
      s0 += __shfl_xor_sync(0xffffffffu, s0, 1);
      s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
      s1 += __shfl_xor_sync(0xffffffffu, s1, 1);
      s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
      const float i0 = __fdividef(1.f, s0), i1 = __fdividef(1.f, s1);
      float o[4][4];
#pragma unroll
      for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int j = 0; j < 4; ++j) o[nt][j] = 0.f;
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {
        uint32_t a[4];
        a[0] = fd_pack_bf16(q0[ks * 4 + 0] * i0, q0[ks * 4 + 1] * i0);
        a[1] = fd_pack_bf16(q1[ks * 4 + 0] * i1, q1[ks * 4 + 1] * i1);
        a[2] = fd_pack_bf16(q0[ks * 4 + 2] * i0, q0[ks * 4 + 3] * i0);
        a[3] = fd_pack_bf16(q1[ks * 4 + 2] * i1, q1[ks * 4 + 3] * i1);
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          const __nv_bfloat16* cr = s_ct + (h * kD + nt * 8 + g) * kCtStride + ks * 16 + 2 * tq;
          mma_bf16(o[nt], a, *reinterpret_cast<const uint32_t*>(cr), *reinterpret_cast<const uint32_t*>(cr + 8));
        }
      }
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        uint8_t* r0 = s_q + (warp * 16 + g) * kApRowBytes + (h * kD + nt * 8 + 2 * tq) * 2;
        *reinterpret_cast<uint32_t*>(r0) = fd_pack_bf16(o[nt][0], o[nt][1]);
        *reinterpret_cast<uint32_t*>(r0 + 8 * kApRowBytes) = fd_pack_bf16(o[nt][2], o[nt][3]);
      }
    }
    __syncwarp();
    // 16 rows x 16 granules per warp -> coalesced 16-byte stores
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int idx = it * 32 + lane;
      const int px = idx >> 4, q16 = idx & 15;
      const int p = p0 + warp * 16 + px;
      if (p < HW)
        *reinterpret_cast<uint4*>(out + ((long)n * HW + p) * kHidden + q16 * 8) =
            *reinterpret_cast<const uint4*>(s_q + (warp * 16 + px) * kApRowBytes + q16 * 16);
    }
  }
}

int la_chunks(int N, int HW, int* chunk_px) {
  // one wave: at most 3 resident blocks per SM (68 KB smem each) in total, chunk a multiple of the tile
  int want = (FD_NUM_SMS * 3) / N;
  if (want < 1) want = 1;
  int px = (HW + want - 1) / want;
  px = ((px + kLaTile - 1) / kLaTile) * kLaTile;
  if (px < kLaTile) px = kLaTile;
  *chunk_px = px;
  return (HW + px - 1) / px;
}

}  // namespace

int fd_attention_tc_launch(const void* qkv, void* out, float* lse, int N, int HW, cudaStream_t st);   // fd_attention_tc.cu

extern "C" {

size_t fd_linattn_workspace_floats(int N, int HW) {
  int px;
  const int chunks = la_chunks(N, HW, &px);
  return (size_t)N * chunks * kLaPartial + (size_t)N * kHeads * kD * kD / 2 + 16;
}

// passes 1 + 2: kv rows = [k(128) | v(128)] bf16, row_stride elements apart -> ctx_t bf16 [N][4][32 e][32 d]
// (softmax over pixels, /HW and the 32^-0.5 q scale folded in)
int fd_linattn_context(const void* kv, int row_stride, void* ctx_t, float* workspace, int N, int HW, void* stream) {
  FD_REQUIRE(kv && ctx_t && workspace && N > 0 && HW > 0 && row_stride >= 2 * kHidden && row_stride % 8 == 0,
             "linattn_context: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  int px;
  const int chunks = la_chunks(N, HW, &px);
  static bool attr_set = false;
  if (!attr_set) {
    FD_CUDA(cudaFuncSetAttribute(linattn_partial_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLaSmemBytes));
    attr_set = true;
  }
  linattn_partial_kernel<<<dim3(chunks, N), 256, kLaSmemBytes, st>>>(static_cast<const __nv_bfloat16*>(kv), row_stride,
                                                                     workspace, HW, px);
  FD_LAUNCH_CHECK();
  linattn_combine_kernel<<<N * kHeads, 1024, 0, st>>>(workspace, static_cast<__nv_bfloat16*>(ctx_t), chunks,
                                                      1.f / (float)HW);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

// fp32 statistics of the k softmax and the context for the backward pass: stats [N][m(128) | Z(128) | ctx(4*32*32)]
int fd_linattn_stats(const void* kv, int row_stride, float* stats, float* workspace, int N, int HW, void* stream) {
  FD_REQUIRE(kv && stats && workspace && N > 0 && HW > 0 && row_stride >= 2 * kHidden && row_stride % 8 == 0,
             "linattn_stats: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  int px;
  const int chunks = la_chunks(N, HW, &px);
  static bool attr_set = false;
  if (!attr_set) {
    FD_CUDA(cudaFuncSetAttribute(linattn_partial_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLaSmemBytes));
    attr_set = true;
  }
  linattn_partial_kernel<<<dim3(chunks, N), 256, kLaSmemBytes, st>>>(static_cast<const __nv_bfloat16*>(kv), row_stride,
                                                                     workspace, HW, px);
  FD_LAUNCH_CHECK();
  linattn_combine_stats_kernel<<<N * kHeads, 1024, 0, st>>>(workspace, stats, chunks, 1.f / (float)HW);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_linattn(const void* qkv, void* out, float* workspace, int N, int HW, void* stream) {
  return fd_linattn_save(qkv, out, nullptr, workspace, N, HW, stream);
}

// fd_linattn that also emits the fp32 statistics of fd_linattn_stats (from the same partial sums) for the backward pass
int fd_linattn_save(const void* qkv, void* out, float* stats, float* workspace, int N, int HW, void* stream) {
  FD_REQUIRE(qkv && out && workspace && N > 0 && HW > 0, "linattn: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  int px;
  const int chunks = la_chunks(N, HW, &px);
  size_t off = (size_t)N * chunks * kLaPartial;
  off = (off + 3) & ~(size_t)3;                                     // 16-byte aligned bf16 ctx^T
  __nv_bfloat16* ctx_t = reinterpret_cast<__nv_bfloat16*>(workspace + off);
  const __nv_bfloat16* q = static_cast<const __nv_bfloat16*>(qkv);
  if (int e = fd_linattn_context(q + kHidden, kQkv, ctx_t, workspace, N, HW, stream)) return e;
  if (stats != nullptr) {
    linattn_combine_stats_kernel<<<N * kHeads, 1024, 0, st>>>(workspace, stats, chunks, 1.f / (float)HW);
    FD_LAUNCH_CHECK();
  }
  int bx = (HW + 63) / 64;
  const int cap = (FD_NUM_SMS * 8 + N - 1) / N;
  if (bx > cap) bx = cap;
  linattn_apply_kernel<<<dim3(bx, N), 128, 0, st>>>(q, ctx_t, static_cast<__nv_bfloat16*>(out), HW);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_attention(const void* qkv, void* out, int N, int HW, void* stream) {
  return fd_attention_lse(qkv, out, nullptr, N, HW, stream);
}

int fd_attention_lse(const void* qkv, void* out, float* lse, int N, int HW, void* stream) {
  FD_REQUIRE(qkv && out && N > 0 && HW > 0, "attention: bad argument");
  FD_REQUIRE(N <= 65535, "attention: batch too large");
  return fd_attention_tc_launch(qkv, out, lse, N, HW, (cudaStream_t)stream);
}

}  // extern "C"
