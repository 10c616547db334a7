// Residual(PreNorm(LinearAttention)) (denoising_diffusion.py:81-87,127-135,216-244) for C in {64, 128} on the 5th-generation
// tensor cores: tcgen05.mma with TMEM accumulators, operands staged by TMA.  Two passes over x and NOTHING else through HBM
// (the unfused form moves LayerNorm(x), the 384-channel qkv tensor and the 128-channel attention output: 13x the bytes).
//
//   y = LayerNorm_g1(x);  q|k|v = W_qkv y;  q = softmax_d(q) 32^-0.5;  k = softmax_pixels(k);  v /= HW
//   ctx[d,e] = sum_p k[p,d] v[p,e]  (per head);  o[p,e] = sum_d ctx[d,e] q[p,d];  out = LayerNorm_g2(W_out o + b) + x
//
// Algebra that removes every intermediate tensor (all exact rewrites of the lines above):
//   * LayerNorm folds into the GEMMs: with W' = W diag(g1), s_j = sum_c W'[j,c],
//       (W y)[p,j] = r_p (sum_c W'[j,c] x[p,c] - mu_p s_j),   mu_p / r_p = mean / rstd of pixel p,
//     so the A operand of the q and k GEMMs is the RAW x tile as TMA lands it; the correction is one FMA in the epilogue.
//   * The softmax over ALL pixels needs no running maximum: |k[p,j]| <= ||W'_j||_2 sqrt(C) because ||y_p||_2 = sqrt(C) after
//     LayerNorm (Cauchy-Schwarz), a weight-only bound m_j.  P[p,d] = exp(k[p,d] - m_d) <= 1 never overflows and the common
//     factor cancels in the normalisation.
//   * v is never formed: sum_p P[p,d] v[p,e] = sum_c W'_v[e,c] G[d,c] with
//       G[d,c] = sum_p (P[p,d] r_p) x[p,c] - T[d],   T[d] = sum_p (P[p,d] r_p) mu_p,   den[d] = sum_p (P[p,d] r_p) sigma_p,
//     i.e. ONE tensor-core GEMM with K = pixels whose B operand is again the raw x tile (pixel rows of 64 channels are the
//     canonical MN-major SWIZZLE_128B layout, as in fd_conv_wgrad.cu); T and den ride on a 16-column GEMM against a tiny
//     tile holding (mu, sigma) split into bf16 hi + lo parts.
//   * to_out folds into the context: o W_out^T = q (ctx W_out^T) = q M, M computed once per sample (128 x C).
//
//   pass 1  linattn_ctx_kernel    x -> per-CTA partial (G, T, den)         [MMA1: k logits, MMA2: P'^T x, P'^T aux]
//           linattn_combine_kernel  partials -> M^T bf16 [N][C][128]         (tiny)
//   pass 2  linattn_apply_kernel  x -> out                                  [MMA1: q logits, MMA2: q_hat M; LayerNorm + x]
//
// Warp roles in both passes (576 threads, one CTA per SM, contiguous tile ranges inside one sample):
//   warp 0 TMA producer, warp 1 TMEM allocator + single-thread tcgen05.mma issuer, warps 2..17 epilogue (TMEM lane quarter =
//   warp % 4; the four warps of a quarter split the columns, 32 each).
#include "fd_tc.cuh"

using namespace fdtc;

namespace {

constexpr int kTilePx = 128;
constexpr int kLaEpiWarps = 16;               // four per TMEM lane quarter: each thread owns 32 of a row's 128 logit columns
constexpr int kLaEpi = kLaEpiWarps * 32;
constexpr int kLaThreads = 64 + kLaEpi;
constexpr float kLog2e = 1.4426950408889634f;

// MN-major SWIZZLE_128B operand (see fd_conv_wgrad.cu): 128-byte rows along M/N, 8 K-rows per 1024-byte atom (SBO),
// successive 64-element M/N chunks `lbo` bytes apart
__device__ __forceinline__ uint64_t la_desc_mn(uint32_t saddr, uint32_t lbo) {
  uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(lbo >> 4) << 16;
  d |= (uint64_t)(1024u >> 4) << 32;
  d |= 1ull << 46;
  d |= 2ull << 61;
  return d;
}
// D fp32, A / B bf16; bit 15 = A is MN-major, bit 16 = B is MN-major
__host__ __device__ constexpr uint32_t la_idesc(int M, int N, bool a_mn, bool b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ float la_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void la_st16(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 la_ld16(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void la_tma_store_3d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(m), "r"(src), "r"(c0),
               "r"(c1), "r"(c2)
               : "memory");
}

// ---- packed fp32x2 arithmetic (FFMA2 / FMUL2 / FADD2 of sm_100): the epilogues are instruction-issue bound
__device__ __forceinline__ uint64_t pk2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ uint64_t pk2u(uint32_t lo, uint32_t hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
  return r;
}
__device__ __forceinline__ float2 up2(uint64_t v) {
  float2 f;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(f.x), "=f"(f.y) : "l"(v));
  return f;
}
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ uint64_t fmul2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t fadd2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

// LayerNorm statistics of a pixel row, shared by the two threads that own the row inside one warp group (`half` 0 / 1): each
// sums half of the row's 16-byte granules, the partial (sum, sum of squares) go through shared memory, the two warps meet on a
// 64-thread named barrier (`bar_id`).  `sx` = [2 halves][128 rows] float2, double buffered by the caller.
template <int C>
__device__ __forceinline__ void la_row_stats2(uint32_t x_tile, int row, int half, int bar_id, float2* sx, float eps, float& mu,
                                              float& r, float& sigma) {
  float s = 0.f, q = 0.f;
#pragma unroll
  for (int gg = 0; gg < C / 16; ++gg) {
    const int g = half * (C / 16) + gg;          // granule of the row: 64-channel chunk g >> 3, 16-byte column g & 7
    // physical column (g ^ row) & 7: the rows a quarter-warp reads in one phase hit different banks
    const uint4 v = la_ld16(x_tile + (g >> 3) * 16384 + row * 128 + (((g & 7) ^ row) & 7) * 16);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = fd_unpack_bf16(w[e]);
      s += f.x + f.y;
      q = fmaf(f.x, f.x, fmaf(f.y, f.y, q));
    }
  }
  sx[half * 128 + row] = make_float2(s, q);
  named_bar_sync(bar_id, 64);
  const float2 o = sx[(half ^ 1) * 128 + row];
  mu = (s + o.x) * (1.f / C);
  const float var = fmaxf((q + o.y) * (1.f / C) - mu * mu, 0.f);
  r = rsqrtf(var + eps);
  sigma = (var + eps) * r;
}

// ------------------------------------------------------------------------------------------------
// weight preparation (once per weight update): rows of to_qkv scaled by the PreNorm gain
//   wq, wk  bf16 [128][C]  = W diag(g1) log2(e)   (the softmaxes use ex2)
//   sq, sk  fp32 [128]     = row sums of the bf16-rounded rows (what the tensor core multiplies)
//   mk      fp32 [128]     = sqrt(C) ||wk_j||_2 (1 + 2^-10): upper bound of the k logit, the softmax shift
//   wv      fp32 [128][C]  = W_v diag(g1)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) linattn_tc_prep_kernel(const float* __restrict__ wqkv, const float* __restrict__ g1,
                                                              __nv_bfloat16* __restrict__ wq, float* __restrict__ sq,
                                                              __nv_bfloat16* __restrict__ wk, float* __restrict__ sk,
                                                              float* __restrict__ mk, float* __restrict__ wv, int C) {
  __shared__ float red[2][4];
  const int j = blockIdx.x;            // row of to_qkv: [q 0..127 | k 128..255 | v 256..383]
  const int t = threadIdx.x;
  float s = 0.f, q2 = 0.f;
  for (int c = t; c < C; c += 128) {
    const float w = wqkv[(long)j * C + c] * g1[c];
    if (j < 256) {
      const __nv_bfloat16 b = __float2bfloat16(w * kLog2e);
      (j < 128 ? wq : wk)[(long)(j & 127) * C + c] = b;
      const float f = __bfloat162float(b);
      s += f;
      q2 = fmaf(f, f, q2);
    } else {
      wv[(long)(j - 256) * C + c] = w;
    }
  }
  s = fd_warp_sum(s);
  q2 = fd_warp_sum(q2);
  if ((t & 31) == 0) {
    red[0][t >> 5] = s;
    red[1][t >> 5] = q2;
  }
  __syncthreads();
  if (t == 0 && j < 256) {
    const float ss = red[0][0] + red[0][1] + red[0][2] + red[0][3];
    const float qq = red[1][0] + red[1][1] + red[1][2] + red[1][3];
    if (j < 128) {
      sq[j] = ss;
    } else {
      sk[j - 128] = ss;
      mk[j - 128] = sqrtf((float)C) * sqrtf(qq) * (1.f + 1.f / 1024.f) + 1e-3f;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// pass 1
// ------------------------------------------------------------------------------------------------
template <int C>
struct CtxCfg {
  static constexpr int kChunks = C / 64;
  static constexpr int kXBytes = kChunks * 16384;          // x tile: 64-channel chunks of [128 px][128 B]
  // deep ring: a slot is held from the TMA load until MMA2 of its tile has retired, i.e. through the whole epilogue; with 4
  // slots only ~2 loads per SM were in flight and the kernel ran at the DRAM latency (4.4 TB/s with ALL work skipped)
  static constexpr int kStages = C == 64 ? 5 : 3;
  static constexpr int kWBytes = kChunks * 16384;          // Wk' [128 rows][C], K-major, 64-channel chunks
  static constexpr int kPBytes = 32768;                    // P' [128 px][128 d]: two 64-d chunks (MN-major A of MMA2)
  static constexpr int kAuxBytes = 4096;                   // aux [16 rows][128 px] K-major: two 64-px chunks of 2 KB
  // P' / aux buffers.  Three (tile i uses buffer i % 3): the group that wrote tile i writes tile i + 2 next, into the buffer
  // tile i - 1 used, whose MMA2 retired before MMA2(i) even started -- so MMA2(i) overlaps the exps of tile i + 2.  With two
  // buffers (one per group) the group waits for its own MMA2 and the two times add up (measured: FD_LA_DBG).
  static constexpr int kNP = C == 64 ? 3 : 2;
  static constexpr int kOffW = kStages * kXBytes;
  static constexpr int kOffP = kOffW + kWBytes;
  static constexpr int kOffAux = kOffP + kNP * kPBytes;
  static constexpr int kOffConst = kOffAux + kNP * kAuxBytes;   // sk[128], -mk[128]
  static constexpr int kOffSx = kOffConst + 1024;             // [2 tile parities][4 parts][128 rows] float2
  static constexpr int kOffBar = kOffSx + 8192;
  static constexpr int kSmemBytes = 1024 + kOffBar + 256;
};

struct CtxParams {
  int N, HW, cps, tiles;      // samples, pixels per sample, CTAs per sample, 128-pixel tiles per sample
  float eps;
  const float* sk;
  const float* mk;
  float* partial;             // [N * cps][128 d][C + 4]: G[d][0..C), T[d], den[d]
  int dbg;                    // FD_LA_DBG & 15 in FD_DIAG builds (results are garbage): 1 skip epilogue math, 2 skip MMA2 + aux, 4 skip row
                              // statistics, 8 skip MMA1
};

template <int C>
__global__ void __launch_bounds__(kLaThreads, 1)
linattn_ctx_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w, const CtxParams p) {
  using Cf = CtxCfg<C>;
  constexpr int S = Cf::kStages;
  constexpr int NCH = Cf::kChunks;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t x_smem = base, w_smem = base + Cf::kOffW, p_smem = base + Cf::kOffP, aux_smem = base + Cf::kOffAux;
  float* s_sk = reinterpret_cast<float*>(gbase + Cf::kOffConst);
  float* s_mk = s_sk + 128;
  const uint32_t bar = base + Cf::kOffBar;
  auto xfull = [&](int s) { return bar + 8u * s; };
  auto xempty = [&](int s) { return bar + 8u * (S + s); };
  const uint32_t wfull = bar + 8u * (2 * S);
  auto d1full = [&](int s) { return bar + 8u * (2 * S + 1 + s); };
  auto d1empty = [&](int s) { return bar + 8u * (2 * S + 3 + s); };
  constexpr int NP = Cf::kNP;
  auto pfull = [&](int s) { return bar + 8u * (2 * S + 5 + s); };
  auto pempty = [&](int s) { return bar + 8u * (2 * S + 5 + NP + s); };
  const uint32_t accfull = bar + 8u * (2 * S + 5 + 2 * NP);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(gbase + Cf::kOffBar + 8 * (2 * S + 6 + 2 * NP));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = blockIdx.x / p.cps, jc = blockIdx.x % p.cps;
  const int t0 = (int)((long)jc * p.tiles / p.cps), t1 = (int)((long)(jc + 1) * p.tiles / p.cps);
  const int nt = t1 - t0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_x);
    tma_prefetch_desc(&map_w);
    for (int s = 0; s < S; ++s) {
      mbar_init(xfull(s), 1);
      mbar_init(xempty(s), 1);
    }
    mbar_init(wfull, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(d1full(s), 1);
      mbar_init(d1empty(s), kLaEpi / 2);       // one warp group (8 warps) owns accumulator stage s
    }
    for (int s = 0; s < NP; ++s) {
      mbar_init(pfull(s), kLaEpi / 2);
      mbar_init(pempty(s), 1);
    }
    mbar_init(accfull, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(s_tmem), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;
  // TMEM columns: D1 (k logits) 2 x 128 at 0 / 128, D2 (G) C columns at 256, D3 (T, den) 16 columns at 384

  if (warp == 0) {
    if (elect_one_sync()) {
      mbar_expect_tx(wfull, Cf::kWBytes);
      for (int ch = 0; ch < NCH; ++ch) tma_load_2d(w_smem + ch * 16384, &map_w, wfull, ch * 64, 0);
      for (int i = 0; i < nt; ++i) {
        const int s = i % S;
        mbar_wait(xempty(s), ((i / S) & 1) ^ 1u);
        mbar_expect_tx(xfull(s), Cf::kXBytes);
        for (int ch = 0; ch < NCH; ++ch)
          tma_load_3d(x_smem + s * Cf::kXBytes + ch * 16384, &map_x, xfull(s), ch * 64, (t0 + i) * kTilePx, n);
      }
    }
  } else if (warp == 1) {
    if (elect_one_sync()) {
      constexpr uint32_t id1 = la_idesc(128, 128, false, false);     // k logits: x (K-major) . Wk'^T (K-major)
      constexpr uint32_t id2 = la_idesc(128, C, true, true);         // G += P'^T (MN-major) . x (MN-major), K = pixels
      constexpr uint32_t id3 = la_idesc(128, 16, true, false);       // T, den += P'^T . aux^T (K-major)
      mbar_wait(wfull, 0);
      const uint64_t wdesc = umma_desc_sw128(w_smem);
      auto mma1 = [&](int i) {
        const int as = i & 1, s = i % S;
        mbar_wait(d1empty(as), ((i >> 1) & 1) ^ 1u);
        mbar_wait(xfull(s), (i / S) & 1);
        tc_fence_after();
        const uint64_t xd = umma_desc_sw128(x_smem + s * Cf::kXBytes);
        if (!(kDiag && (p.dbg & 8))) {
#pragma unroll
          for (int ch = 0; ch < NCH; ++ch)
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(tmem_base + as * 128, xd + (uint64_t)(ch * 1024 + 2 * k), wdesc + (uint64_t)(ch * 1024 + 2 * k), id1,
                        (ch | k) != 0 ? 1u : 0u);
        }
        umma_commit(d1full(as));
      };
      if (nt > 0) mma1(0);
      for (int i = 0; i < nt; ++i) {
        if (i + 1 < nt) mma1(i + 1);
        const int pb = i % NP, s = i % S;
        mbar_wait(pfull(pb), (i / NP) & 1);
        tc_fence_after();
        const uint64_t pd = la_desc_mn(p_smem + pb * Cf::kPBytes, 16384);
        const uint64_t xd = la_desc_mn(x_smem + s * Cf::kXBytes, 16384);
        const uint64_t ad = umma_desc_sw128(aux_smem + pb * Cf::kAuxBytes);
        if (!(kDiag && (p.dbg & 2))) {
#pragma unroll
          for (int ks = 0; ks < 8; ++ks)       // 16 pixels per step = two 8-pixel atoms = 2048 B
            umma_bf16(tmem_base + 256, pd + (uint64_t)(ks * 128), xd + (uint64_t)(ks * 128), id2, (i | ks) != 0 ? 1u : 0u);
#pragma unroll
          for (int ks = 0; ks < 8; ++ks)
            umma_bf16(tmem_base + 384, pd + (uint64_t)(ks * 128), ad + (uint64_t)((ks >> 2) * 128 + 2 * (ks & 3)), id3,
                      (i | ks) != 0 ? 1u : 0u);
        }
        umma_commit(xempty(s));
        umma_commit(pempty(pb));
      }
      umma_commit(accfull);
    }
    __syncwarp();
  } else {
    // ===================== epilogue warps 2..17: two groups of 8 warps on alternating tiles =====================
    // The exp of 128 x 128 logits per tile keeps the MUFU pipe busy for 1024 cycles; everything else a tile needs (row
    // statistics, TMEM loads, barrier round trips) overlaps it only if ANOTHER tile's exps are in flight meanwhile (measured
    // with FD_LA_DBG: with one group the parts simply add up).  Group g owns tiles i = g (mod 2), i.e. accumulator stage g
    // and P' buffer g.  Inside a group the two warps of a TMEM lane quarter split a row's 128 logit columns (2 heads each).
    const int et = threadIdx.x - 64, ew = warp - 2;
    const int grp = ew >> 3, half = (ew >> 2) & 1, quarter = warp & 3;
    const int part = ew >> 2;                                  // 0..3, used for the final accumulator read-out only
    const int row = quarter * 32 + lane;
    if (et < 128) s_sk[et] = __ldg(p.sk + et);
    else if (et < 256) s_mk[et - 128] = -__ldg(p.mk + et - 128);
    for (int i = et; i < NP * Cf::kAuxBytes / 16; i += kLaEpi) la_st16(aux_smem + i * 16, 0u, 0u, 0u, 0u);   // rows 4..15 stay zero
    named_bar_sync(1, kLaEpi);
    float2* s_sx = reinterpret_cast<float2*>(gbase + Cf::kOffSx) + grp * 512;       // [group][use parity][half][row]
    const uint32_t lane_off = (uint32_t)(quarter * 32) << 16;
    const int as = grp;
    for (int i = grp; i < nt; i += 2) {
      const int s = i % S, u = i >> 1, pb = i % NP;
      mbar_wait(xfull(s), (i / S) & 1);
      float mu = 0.f, r = 1.f, sigma = 1.f;
      if (!(kDiag && (p.dbg & 4)))
        la_row_stats2<C>(x_smem + s * Cf::kXBytes, row, half, 4 + grp * 4 + quarter, s_sx + (u & 1) * 256, p.eps, mu, r, sigma);
      const bool valid = (t0 + i) * kTilePx + row < p.HW;
      const uint64_t nrm2 = pk2(-r * mu, -r * mu), r2 = pk2(r, r);
      const uint64_t rv2 = valid ? r2 : 0ull;
      mbar_wait(pempty(pb), ((i / NP) & 1) ^ 1u);
      mbar_wait(d1full(as), u & 1);
      tc_fence_after();
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const int col0 = half * 64 + cc * 32;
        uint32_t acc[32];
        tmem_ld32(tmem_base + lane_off + (uint32_t)(as * 128 + col0), acc);
        tmem_ld_wait();
        if (cc == 1) {
          tc_fence_before();
          mbar_arrive(d1empty(as));
        }
        if (kDiag && (p.dbg & 1)) continue;
        uint32_t pk[16];
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const ulonglong2 s4 = *reinterpret_cast<const ulonglong2*>(s_sk + col0 + j4 * 4);
          const ulonglong2 m4 = *reinterpret_cast<const ulonglong2*>(s_mk + col0 + j4 * 4);
          // k' - m = r acc - r mu s_j - m_j  (log2 e folded into Wk'); P' = exp2(.) r_p, zero for rows past the sample
          const float2 a0 = up2(ffma2(r2, pk2u(acc[j4 * 4 + 0], acc[j4 * 4 + 1]), ffma2(nrm2, s4.x, m4.x)));
          const float2 a1 = up2(ffma2(r2, pk2u(acc[j4 * 4 + 2], acc[j4 * 4 + 3]), ffma2(nrm2, s4.y, m4.y)));
          const float2 p0 = up2(fmul2(pk2(la_ex2(a0.x), la_ex2(a0.y)), rv2));
          const float2 p1 = up2(fmul2(pk2(la_ex2(a1.x), la_ex2(a1.y)), rv2));
          pk[j4 * 2] = fd_pack_bf16(p0.x, p0.y);
          pk[j4 * 2 + 1] = fd_pack_bf16(p1.x, p1.y);
        }
        const uint32_t rbase = p_smem + pb * Cf::kPBytes + half * 16384 + row * 128;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint32_t piece = (uint32_t)(cc * 4 + q) ^ (uint32_t)(row & 7);
          la_st16(rbase + piece * 16u, pk[q * 4], pk[q * 4 + 1], pk[q * 4 + 2], pk[q * 4 + 3]);
        }
      }
      {
        // aux tile, K-major [16 rows][64 px] per 64-pixel chunk: rows 0/1 = mu hi/lo (written by half 0), 2/3 = sigma hi/lo
        const float val = half == 0 ? mu : sigma;
        const __nv_bfloat16 hi = __float2bfloat16(val);
        const __nv_bfloat16 lo = __float2bfloat16(val - __bfloat162float(hi));
        const uint32_t abase = aux_smem + pb * Cf::kAuxBytes + (row >> 6) * 2048 + (row & 7) * 2;
        const int g = (row & 63) >> 3;
        const int r0 = half * 2, r1 = half * 2 + 1;
        asm volatile("st.shared.b16 [%0], %1;" ::"r"(abase + r0 * 128 + ((g ^ r0) & 7) * 16), "h"(*reinterpret_cast<const uint16_t*>(&hi))
                     : "memory");
        asm volatile("st.shared.b16 [%0], %1;" ::"r"(abase + r1 * 128 + ((g ^ r1) & 7) * 16), "h"(*reinterpret_cast<const uint16_t*>(&lo))
                     : "memory");
      }
      fence_proxy_async_smem();
      mbar_arrive(pfull(pb));
    }
    // ---- the CTA's accumulators -> its partial
    mbar_wait(accfull, 0);
    tc_fence_after();
    float* out = p.partial + ((long)blockIdx.x * 128 + row) * (C + 4);
    if (part < C / 32) {
      uint32_t acc[32];
      tmem_ld32(tmem_base + lane_off + (uint32_t)(256 + part * 32), acc);
      tmem_ld_wait();
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4)
        *reinterpret_cast<float4*>(out + part * 32 + j4 * 4) =
            make_float4(__uint_as_float(acc[j4 * 4]), __uint_as_float(acc[j4 * 4 + 1]), __uint_as_float(acc[j4 * 4 + 2]),
                        __uint_as_float(acc[j4 * 4 + 3]));
    }
    if (part == 3) {
      uint32_t acc[16];
      tmem_ld16(tmem_base + lane_off + 384u, acc);       // columns 0..3 = T hi/lo, den hi/lo parts
      tmem_ld_wait();
      *reinterpret_cast<float4*>(out + C) = make_float4(__uint_as_float(acc[0]) + __uint_as_float(acc[1]),
                                                        __uint_as_float(acc[2]) + __uint_as_float(acc[3]), 0.f, 0.f);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------
// combine: partials of one (sample, head) -> M^T[co][d] = sum_{e in head(d)} ctx[d][e] W_out[co][e]   (bf16 [N][C][128])
//   ctx[d][e] = 32^-0.5 / (HW den[d]) sum_c (G[d][c] - T[d]) W'_v[e][c]
// grid (N, 4 heads), 256 threads; partials are added in a fixed order (run-to-run bit-stable)
// ------------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(256) linattn_tc_combine_kernel(const float* __restrict__ partial, const float* __restrict__ wv,
                                                                 const float* __restrict__ wout, __nv_bfloat16* __restrict__ mt,
                                                                 int cps, int HW) {
  __shared__ float s_g[32][C + 1];
  __shared__ float s_wv[32][C + 1];
  __shared__ float s_ctx[32][33];
  __shared__ float s_T[32], s_den[32];
  const int n = blockIdx.x, head = blockIdx.y, t = threadIdx.x;
  constexpr int V4 = (C + 4) / 4;
  for (int idx = t; idx < 32 * V4; idx += 256) {
    const int dd = idx / V4, v = idx - dd * V4;
    // six loads in flight per thread, six accumulators combined in a fixed order: one dependent load after another over the
    // ~18 CTAs of a sample made this kernel pure L2 latency (34 us per launch for 3 MB of partials)
    constexpr int U = 6;
    float4 acc[U];
#pragma unroll
    for (int u = 0; u < U; ++u) acc[u] = make_float4(0.f, 0.f, 0.f, 0.f);
    const float* src = partial + (((long)n * cps) * 128 + head * 32 + dd) * (C + 4) + v * 4;
    constexpr long kStep = 128L * (C + 4);
    int j = 0;
    for (; j + U <= cps; j += U) {
      float4 x[U];
#pragma unroll
      for (int u = 0; u < U; ++u) x[u] = *reinterpret_cast<const float4*>(src + (long)(j + u) * kStep);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        acc[u].x += x[u].x;
        acc[u].y += x[u].y;
        acc[u].z += x[u].z;
        acc[u].w += x[u].w;
      }
    }
    for (int u = 0; j < cps; ++j, ++u) {
      const float4 x = *reinterpret_cast<const float4*>(src + (long)j * kStep);
      acc[u].x += x.x;
      acc[u].y += x.y;
      acc[u].z += x.z;
      acc[u].w += x.w;
    }
    float4 a;
    a.x = ((acc[0].x + acc[1].x) + (acc[2].x + acc[3].x)) + (acc[4].x + acc[5].x);
    a.y = ((acc[0].y + acc[1].y) + (acc[2].y + acc[3].y)) + (acc[4].y + acc[5].y);
    a.z = ((acc[0].z + acc[1].z) + (acc[2].z + acc[3].z)) + (acc[4].z + acc[5].z);
    a.w = ((acc[0].w + acc[1].w) + (acc[2].w + acc[3].w)) + (acc[4].w + acc[5].w);
    if (v < C / 4) {
      s_g[dd][v * 4] = a.x;
      s_g[dd][v * 4 + 1] = a.y;
      s_g[dd][v * 4 + 2] = a.z;
      s_g[dd][v * 4 + 3] = a.w;
    } else {
      s_T[dd] = a.x;
      s_den[dd] = a.y;
    }
  }
  for (int idx = t; idx < 32 * C; idx += 256) {
    const int e = idx / C, c = idx - e * C;
    s_wv[e][c] = __ldg(wv + (long)(head * 32 + e) * C + c);
  }
  __syncthreads();
  for (int o = t; o < 1024; o += 256) {
    const int dd = o >> 5, e = o & 31;
    const float T = s_T[dd];
    float a = 0.f;
#pragma unroll 8
    for (int c = 0; c < C; ++c) a = fmaf(s_g[dd][c] - T, s_wv[e][c], a);
    // 32^-0.5 (q scale, :238), 1 / HW (v, :240), softmax denominator
    s_ctx[dd][e] = a * (0.17677669529663687f / (s_den[dd] * (float)HW));
  }
  __syncthreads();
  for (int o = t; o < 32 * C; o += 256) {
    const int dd = o & 31, co = o >> 5;
    const float* w = wout + (long)co * 128 + head * 32;
    float a = 0.f;
#pragma unroll
    for (int e = 0; e < 32; ++e) a = fmaf(s_ctx[dd][e], __ldg(w + e), a);
    mt[((long)n * C + co) * 128 + head * 32 + dd] = __float2bfloat16(a);
  }
}

// ------------------------------------------------------------------------------------------------
// pass 2
// ------------------------------------------------------------------------------------------------
template <int C>
struct ApTcCfg {
  static constexpr int kChunks = C / 64;
  static constexpr int kXBytes = kChunks * 16384;
  static constexpr int kStages = C == 64 ? 6 : 2;
  static constexpr int kWBytes = kChunks * 16384;          // Wq' [128 rows][C]
  static constexpr int kMBytes = 2 * C * 128;              // M^T [C rows][128 d]: two 64-d chunks of [C][128 B]
  static constexpr int kQBytes = 32768;                    // q_hat [128 px][128 d]: two 64-d chunks (K-major A of MMA2)
  static constexpr int kNQ = C == 64 ? 2 : 1;
  static constexpr int kOBytes = kChunks * 16384;          // output staging: one 64-channel slab per chunk
  static constexpr int kNO = 1;
  static constexpr int kOffW = kStages * kXBytes;
  static constexpr int kOffM = kOffW + kWBytes;
  static constexpr int kOffQ = kOffM + kMBytes;
  static constexpr int kOffO = kOffQ + kNQ * kQBytes;
  static constexpr int kOffConst = kOffO + kNO * kOBytes;    // sq[128], bout[C], g2[C]  (<= 1.5 KB)
  static constexpr int kOffSx = kOffConst + 2048;            // partial-sum exchange of the output group: [2 uses][2 parities][2][128] float2
  static constexpr int kOffRs = kOffSx + 8192;               // (mu, rstd) of x per row, [2 tile parities][128] float2
  static constexpr int kOffBar = kOffRs + 2048;
  static constexpr int kSmemBytes = 1024 + kOffBar + 256;
};

struct ApParams {
  int N, HW, cps, tiles;
  float eps;
  const float* sq;
  const float* bout;
  const float* g2;
  int dbg;                    // FD_LA_DBG >> 4 in FD_DIAG builds (results are garbage)
};

template <int C>
__global__ void __launch_bounds__(kLaThreads, 1)
linattn_apply_kernel_tc(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                        const __grid_constant__ CUtensorMap map_m, const __grid_constant__ CUtensorMap map_out, const ApParams p) {
  using Cf = ApTcCfg<C>;
  constexpr int S = Cf::kStages;
  constexpr int NCH = Cf::kChunks;
  constexpr int NQ = Cf::kNQ;
  constexpr int NO = Cf::kNO;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t x_smem = base, w_smem = base + Cf::kOffW, m_smem = base + Cf::kOffM, q_smem = base + Cf::kOffQ,
                 o_smem = base + Cf::kOffO;
  float* s_sq = reinterpret_cast<float*>(gbase + Cf::kOffConst);
  float* s_b = s_sq + 128;
  float* s_g2 = s_b + C;
  float2* s_sx = reinterpret_cast<float2*>(gbase + Cf::kOffSx);      // [softmax | output group][tile parity][half][row]
  const uint32_t bar = base + Cf::kOffBar;
  auto xfull = [&](int s) { return bar + 8u * s; };
  auto xempty = [&](int s) { return bar + 8u * (S + s); };
  const uint32_t wfull = bar + 8u * (2 * S);
  auto d1full = [&](int s) { return bar + 8u * (2 * S + 1 + s); };
  auto d1empty = [&](int s) { return bar + 8u * (2 * S + 3 + s); };
  auto qfull = [&](int s) { return bar + 8u * (2 * S + 5 + s); };
  auto qempty = [&](int s) { return bar + 8u * (2 * S + 7 + s); };
  auto d2full = [&](int s) { return bar + 8u * (2 * S + 9 + s); };
  auto d2empty = [&](int s) { return bar + 8u * (2 * S + 11 + s); };
  auto sfull = [&](int s) { return bar + 8u * (2 * S + 13 + s); };
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(gbase + Cf::kOffBar + 8 * (2 * S + 15));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = blockIdx.x / p.cps, jc = blockIdx.x % p.cps;
  const int t0 = (int)((long)jc * p.tiles / p.cps), t1 = (int)((long)(jc + 1) * p.tiles / p.cps);
  const int nt = t1 - t0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_x);
    tma_prefetch_desc(&map_w);
    tma_prefetch_desc(&map_m);
    tma_prefetch_desc(&map_out);
    for (int s = 0; s < S; ++s) {
      mbar_init(xfull(s), 1);
      mbar_init(xempty(s), kLaEpi / 2);        // the output group is the only reader of the x tile besides the tensor core
    }
    mbar_init(wfull, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(sfull(s), kLaEpi / 2);
      mbar_init(d1full(s), 1);
      mbar_init(d1empty(s), kLaEpi / 2);       // softmax group (warps 2..9)
      mbar_init(qfull(s), kLaEpi / 2);
      mbar_init(qempty(s), 1);
      mbar_init(d2full(s), 1);
      mbar_init(d2empty(s), kLaEpi / 2);       // output group (warps 10..17)
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(s_tmem), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;
  // TMEM columns: D1 (q logits) 2 x 128 at 0 / 128, D2 (q_hat M) 2 x C at 256 / 384

  if (warp == 0) {
    if (elect_one_sync()) {
      mbar_expect_tx(wfull, Cf::kWBytes + Cf::kMBytes);
      for (int ch = 0; ch < NCH; ++ch) tma_load_2d(w_smem + ch * 16384, &map_w, wfull, ch * 64, 0);
      for (int dc = 0; dc < 2; ++dc) tma_load_3d(m_smem + dc * (C * 128), &map_m, wfull, dc * 64, 0, n);
      for (int i = 0; i < nt; ++i) {
        const int s = i % S;
        mbar_wait(xempty(s), ((i / S) & 1) ^ 1u);
        mbar_expect_tx(xfull(s), Cf::kXBytes);
        for (int ch = 0; ch < NCH; ++ch)
          tma_load_3d(x_smem + s * Cf::kXBytes + ch * 16384, &map_x, xfull(s), ch * 64, (t0 + i) * kTilePx, n);
      }
    }
  } else if (warp == 1) {
    if (elect_one_sync()) {
      constexpr uint32_t id1 = la_idesc(128, 128, false, false);
      constexpr uint32_t id2 = la_idesc(128, C, false, false);
      mbar_wait(wfull, 0);
      const uint64_t wdesc = umma_desc_sw128(w_smem), mdesc = umma_desc_sw128(m_smem);
      auto mma1 = [&](int i) {
        const int as = i & 1, s = i % S;
        mbar_wait(d1empty(as), ((i >> 1) & 1) ^ 1u);
        mbar_wait(xfull(s), (i / S) & 1);
        tc_fence_after();
        const uint64_t xd = umma_desc_sw128(x_smem + s * Cf::kXBytes);
        if (!(kDiag && (p.dbg & 8))) {
#pragma unroll
          for (int ch = 0; ch < NCH; ++ch)
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(tmem_base + as * 128, xd + (uint64_t)(ch * 1024 + 2 * k), wdesc + (uint64_t)(ch * 1024 + 2 * k), id1,
                        (ch | k) != 0 ? 1u : 0u);
        }
        umma_commit(d1full(as));
      };
      if (nt > 0) mma1(0);
      for (int i = 0; i < nt; ++i) {
        if (i + 1 < nt) mma1(i + 1);
        const int qb = i % NQ, as = i & 1;
        mbar_wait(qfull(qb), (i / NQ) & 1);
        mbar_wait(d2empty(as), ((i >> 1) & 1) ^ 1u);
        tc_fence_after();
        const uint64_t qd = umma_desc_sw128(q_smem + qb * Cf::kQBytes);
        if (!(kDiag && (p.dbg & 2))) {
#pragma unroll
          for (int ks = 0; ks < 8; ++ks)       // K = 128 d: two 64-d chunks x four 16-element steps
            umma_bf16(tmem_base + 256 + as * 128, qd + (uint64_t)((ks >> 2) * 1024 + 2 * (ks & 3)),
                      mdesc + (uint64_t)((ks >> 2) * (C * 128 >> 4) + 2 * (ks & 3)), id2, ks != 0 ? 1u : 0u);
        }
        umma_commit(d2full(as));
        umma_commit(qempty(qb));
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue warps 2..17: softmax group (2..9) and output group (10..17) =====================
    // The two epilogues of a tile are bound by different pipes (softmax: MUFU, 128 x 128 exps; output: FMA + shared memory), so
    // they run CONCURRENTLY on different warps, one tile apart, coupled only through the mbarriers (measured with FD_LA_DBG:
    // run back to back by the same warps their times add up).  Inside a group the two warps of a TMEM lane quarter split the
    // row's columns and exchange their partial row statistics through shared memory on a 64-thread named barrier.
    const int ew = warp - 2, et = threadIdx.x - 64;
    const int grp = ew >> 3, half = (ew >> 2) & 1, quarter = warp & 3;
    const int row = quarter * 32 + lane;
    for (int i = et; i < 128 + 2 * C; i += kLaEpi)
      s_sq[i] = i < 128 ? __ldg(p.sq + i) : (i < 128 + C ? __ldg(p.bout + i - 128) : __ldg(p.g2 + i - 128 - C));
    named_bar_sync(1, kLaEpi);
    const uint32_t lane_off = (uint32_t)(quarter * 32) << 16;

    float2* s_rs = reinterpret_cast<float2*>(gbase + Cf::kOffRs);
    if (grp == 0) {
      // ---- q logits -> softmax over d per head -> q_hat tile (K-major A operand of MMA2).  The row statistics of x come from
      // the output group (it has the slack); both heads of a thread are processed interleaved (64 independent exps in flight).
      for (int i = 0; i < nt; ++i) {
        const int qb = i % NQ, as = i & 1;
        mbar_wait(sfull(i & 1), (i >> 1) & 1);
        const float2 st = s_rs[(i & 1) * 128 + row];
        const float r = st.y;
        const uint64_t nrm2 = pk2(-r * st.x, -r * st.x), r2 = pk2(r, r);
        mbar_wait(qempty(qb), ((i / NQ) & 1) ^ 1u);
        mbar_wait(d1full(as), (i >> 1) & 1);
        tc_fence_after();
        uint32_t acc[2][32];
        tmem_ld32(tmem_base + lane_off + (uint32_t)(as * 128 + half * 64), acc[0]);
        tmem_ld32(tmem_base + lane_off + (uint32_t)(as * 128 + half * 64 + 32), acc[1]);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(d1empty(as));
        if (kDiag && (p.dbg & 1)) {
          fence_proxy_async_smem();
          mbar_arrive(qfull(qb));
          continue;
        }
        float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int col0 = (half * 2 + hh) * 32;        // one head = 32 columns
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const ulonglong2 s4 = *reinterpret_cast<const ulonglong2*>(s_sq + col0 + j4 * 4);
            const float2 a0 = up2(ffma2(r2, pk2u(acc[hh][j4 * 4 + 0], acc[hh][j4 * 4 + 1]), fmul2(nrm2, s4.x)));
            const float2 a1 = up2(ffma2(r2, pk2u(acc[hh][j4 * 4 + 2], acc[hh][j4 * 4 + 3]), fmul2(nrm2, s4.y)));
            acc[hh][j4 * 4 + 0] = __float_as_uint(a0.x);
            acc[hh][j4 * 4 + 1] = __float_as_uint(a0.y);
            acc[hh][j4 * 4 + 2] = __float_as_uint(a1.x);
            acc[hh][j4 * 4 + 3] = __float_as_uint(a1.y);
            mx[hh] = fmaxf(mx[hh], fmaxf(fmaxf(a0.x, a0.y), fmaxf(a1.x, a1.y)));
          }
        }
        float sum[2] = {0.f, 0.f};
#pragma unroll
        for (int j = 0; j < 32; ++j) {
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            const float e = la_ex2(__uint_as_float(acc[hh][j]) - mx[hh]);
            acc[hh][j] = __float_as_uint(e);
            sum[hh] += e;
          }
        }
        const uint32_t rbase = q_smem + qb * Cf::kQBytes + half * 16384 + row * 128;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const float inv = __fdividef(1.f, sum[hh]);
          const uint64_t inv2 = pk2(inv, inv);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            uint32_t w[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 f = up2(fmul2(pk2u(acc[hh][q * 8 + e * 2], acc[hh][q * 8 + e * 2 + 1]), inv2));
              w[e] = fd_pack_bf16(f.x, f.y);
            }
            const uint32_t piece = (uint32_t)(hh * 4 + q) ^ (uint32_t)(row & 7);
            la_st16(rbase + piece * 16u, w[0], w[1], w[2], w[3]);
          }
        }
        fence_proxy_async_smem();
        mbar_arrive(qfull(qb));
      }
    } else {
      // ---- q_hat M + b -> LayerNorm_g2 -> + x -> bf16 -> TMA store
      constexpr int CPT = C / 2;           // output channels per thread (32 or 64)
      const int gw = ew - 8;               // 0..7 inside the group
      const int col0 = half * CPT;
      uint32_t slab_count = 0;
      // LayerNorm statistics of the x rows for the softmax group, one tile ahead of this group's own work.  No "empty"
      // barrier is needed for s_rs: statistics of tile j + 2 are written after this group finished the output of tile j,
      // which needed MMA2(j), which needed the softmax group to be done with tile j (and its statistics).
      auto x_stats = [&](int j) {
        const int sj = j % S;
        mbar_wait(xfull(sj), (j / S) & 1);
        float mu = 0.f, r = 1.f, sigma = 1.f;
        if (!(kDiag && (p.dbg & 4))) la_row_stats2<C>(x_smem + sj * Cf::kXBytes, row, half, 8 + quarter, s_sx + (j & 1) * 256, p.eps, mu, r, sigma);
        if (half == 0) s_rs[(j & 1) * 128 + row] = make_float2(mu, r);
        mbar_arrive(sfull(j & 1));
      };
      if (nt > 0) x_stats(0);
      for (int i = 0; i < nt; ++i) {
        const int s = i % S, as = i & 1;
        if (i + 1 < nt) x_stats(i + 1);
        mbar_wait(d2full(as), (i >> 1) & 1);
        tc_fence_after();
        uint64_t o[CPT / 2];
        uint64_t sm2 = 0ull, sq22 = 0ull;
#pragma unroll
        for (int cb = 0; cb < CPT / 32; ++cb) {
          uint32_t acc[32];
          tmem_ld32(tmem_base + lane_off + (uint32_t)(256 + as * 128 + col0 + cb * 32), acc);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const uint64_t x = fadd2(pk2u(acc[2 * j], acc[2 * j + 1]), *reinterpret_cast<const uint64_t*>(s_b + col0 + cb * 32 + 2 * j));
            o[cb * 16 + j] = x;
            sm2 = fadd2(sm2, x);
            sq22 = ffma2(x, x, sq22);
          }
        }
        tc_fence_before();
        mbar_arrive(d2empty(as));
        const uint32_t ob = slab_count % NO;
        ++slab_count;
        if (kDiag && (p.dbg & 16)) {
          mbar_arrive(xempty(s));
          continue;
        }
        const float2 smf = up2(sm2), sqf = up2(sq22);
        const float sm = smf.x + smf.y, sq2 = sqf.x + sqf.y;
        float2* sx = s_sx + 512 + (i & 1) * 256;
        sx[half * 128 + row] = make_float2(sm, sq2);
        if (gw == 0 && elect_one_sync()) tma_store_wait_read<NO - 1>();      // the store that last used this staging buffer has read it
        named_bar_sync(2, kLaEpi / 2);       // (also orders the statistics exchange: all 8 warps are past their stores to sx)
        const float2 other = sx[(half ^ 1) * 128 + row];
        const float mean = (sm + other.x) * (1.f / C);
        const float var = fmaxf((sq2 + other.y) * (1.f / C) - mean * mean, 0.f);
        const float rstd = rsqrtf(var + p.eps);
        const uint64_t rstd2 = pk2(rstd, rstd), nmr2 = pk2(-mean * rstd, -mean * rstd);
#pragma unroll
        for (int cb = 0; cb < CPT / 32; ++cb) {
          const int c0 = col0 + cb * 32;       // absolute output channel of o[cb * 16]
          const int chunk = c0 >> 6, g0 = (c0 & 63) >> 3;
          const uint32_t xrow = x_smem + s * Cf::kXBytes + chunk * 16384 + row * 128;
          const uint32_t orow = o_smem + ob * Cf::kOBytes + chunk * 16384 + row * 128;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint32_t piece = (uint32_t)(g0 + q) ^ (uint32_t)(row & 7);
            const uint4 xr = la_ld16(xrow + piece * 16u);
            const uint32_t xw[4] = {xr.x, xr.y, xr.z, xr.w};
            uint32_t ow[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 f = fd_unpack_bf16(xw[e]);
              // ((o - mean) rstd) g2 + x
              const uint64_t nrm = ffma2(o[cb * 16 + q * 4 + e], rstd2, nmr2);
              const float2 y = up2(ffma2(nrm, *reinterpret_cast<const uint64_t*>(s_g2 + c0 + q * 8 + e * 2), pk2(f.x, f.y)));
              ow[e] = fd_pack_bf16(y.x, y.y);
            }
            la_st16(orow + piece * 16u, ow[0], ow[1], ow[2], ow[3]);
          }
        }
        fence_proxy_async_smem();
        mbar_arrive(xempty(s));              // this group's reads of the x tile (the residual) are done
        named_bar_sync(3, kLaEpi / 2);
        if (gw == 0 && elect_one_sync() && !(kDiag && (p.dbg & 32))) {
          for (int ch = 0; ch < NCH; ++ch)
            la_tma_store_3d(&map_out, o_smem + ob * Cf::kOBytes + ch * 16384, ch * 64, (t0 + i) * kTilePx, n);
          tma_store_commit();
        }
      }
      __syncwarp();
      if (gw == 0 && elect_one_sync()) tma_store_wait_all();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

int ctas_per_sample(int N, int tiles) {
  int cps = FD_NUM_SMS / N;
  if (cps < 1) cps = 1;
  if (cps > tiles) cps = tiles;
  return cps;
}

template <int C>
int run_tc(const void* x, const void* wk, const float* sk, const float* mk, const void* wq, const float* sq, const float* wv,
           const float* wout, const float* bout, const float* g2, void* out, float* workspace, int N, int HW, float eps,
           cudaStream_t st) {
  const int tiles = (HW + kTilePx - 1) / kTilePx;
  const int cps = ctas_per_sample(N, tiles);
  float* partial = workspace;
  __nv_bfloat16* mt = reinterpret_cast<__nv_bfloat16*>(workspace + (size_t)N * cps * 128 * (C + 4));
  CUtensorMap map_x, map_wk, map_wq, map_m, map_out;
  {
    const uint64_t dims[3] = {(uint64_t)C, (uint64_t)HW, (uint64_t)N};
    const uint64_t str[2] = {(uint64_t)C * 2, (uint64_t)HW * C * 2};
    const uint32_t box[3] = {64, (uint32_t)kTilePx, 1};
    if (int e = make_tmap_bf16(&map_x, x, 3, dims, str, box)) return e;
    if (int e = make_tmap_bf16(&map_out, out, 3, dims, str, box)) return e;
  }
  {
    const uint64_t dims[2] = {(uint64_t)C, 128};
    const uint64_t str[1] = {(uint64_t)C * 2};
    const uint32_t box[2] = {64, 128};
    if (int e = make_tmap_bf16(&map_wk, wk, 2, dims, str, box)) return e;
    if (int e = make_tmap_bf16(&map_wq, wq, 2, dims, str, box)) return e;
  }
  {
    const uint64_t dims[3] = {128, (uint64_t)C, (uint64_t)N};
    const uint64_t str[2] = {256, (uint64_t)C * 256};
    const uint32_t box[3] = {64, (uint32_t)C, 1};
    if (int e = make_tmap_bf16(&map_m, mt, 3, dims, str, box)) return e;
  }
  static bool attr_set = false;
  if (!attr_set) {
    FD_CUDA(cudaFuncSetAttribute(linattn_ctx_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, CtxCfg<C>::kSmemBytes));
    FD_CUDA(cudaFuncSetAttribute(linattn_apply_kernel_tc<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, ApTcCfg<C>::kSmemBytes));
    attr_set = true;
  }
  static const int la_dbg = fd_diag_bits("FD_LA_DBG");
  CtxParams cp{N, HW, cps, tiles, eps, sk, mk, partial, la_dbg & 15};
  linattn_ctx_kernel<C><<<N * cps, kLaThreads, CtxCfg<C>::kSmemBytes, st>>>(map_x, map_wk, cp);
  FD_LAUNCH_CHECK();
  linattn_tc_combine_kernel<C><<<dim3(N, 4), 256, 0, st>>>(partial, wv, wout, mt, cps, HW);
  FD_LAUNCH_CHECK();
  ApParams ap{N, HW, cps, tiles, eps, sq, bout, g2, la_dbg >> 4};
  linattn_apply_kernel_tc<C><<<N * cps, kLaThreads, ApTcCfg<C>::kSmemBytes, st>>>(map_x, map_wq, map_m, map_out, ap);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

}  // namespace

extern "C" {

size_t fd_linattn_tc_workspace_floats(int N, int HW, int C) {
  const int tiles = (HW + kTilePx - 1) / kTilePx;
  const int cps = ctas_per_sample(N > 0 ? N : 1, tiles > 0 ? tiles : 1);
  return (size_t)N * cps * 128 * (C + 4) + (size_t)N * C * 128 / 2 + 64;
}

int fd_linattn_tc_prep(const float* wqkv, const float* g1, void* wq, float* sq, void* wk, float* sk, float* mk, float* wv, int C,
                       void* stream) {
  FD_REQUIRE(wqkv && g1 && wq && sq && wk && sk && mk && wv, "linattn_tc_prep: null pointer");
  FD_REQUIRE(C == 64 || C == 128, "linattn_tc_prep: C=%d not in {64,128}", C);
  linattn_tc_prep_kernel<<<384, 128, 0, (cudaStream_t)stream>>>(wqkv, g1, static_cast<__nv_bfloat16*>(wq), sq,
                                                               static_cast<__nv_bfloat16*>(wk), sk, mk, wv, C);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_linattn_tc(const void* x, const void* wk, const float* sk, const float* mk, const void* wq, const float* sq,
                  const float* wv, const float* wout, const float* bout, const float* g2, void* out, float* workspace, int N,
                  int HW, int C, float eps, void* stream) {
  FD_REQUIRE(x && wk && sk && mk && wq && sq && wv && wout && bout && g2 && out && workspace, "linattn_tc: null pointer");
  FD_REQUIRE(N > 0 && HW > 0, "linattn_tc: bad geometry N=%d HW=%d", N, HW);
  FD_REQUIRE(C == 64 || C == 128, "linattn_tc: C=%d not in {64,128}", C);
  cudaStream_t st = (cudaStream_t)stream;
  if (C == 64) return run_tc<64>(x, wk, sk, mk, wq, sq, wv, wout, bout, g2, out, workspace, N, HW, eps, st);
  return run_tc<128>(x, wk, sk, mk, wq, sq, wv, wout, bout, g2, out, workspace, N, HW, eps, st);
}

}  // extern "C"
