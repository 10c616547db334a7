// Implicit-GEMM convolution on the 5th-generation tensor cores (tcgen05 + TMEM), operands staged
// by TMA.  Replaces every nn.Conv2d / WeightStandardizedConv2d call of the reference UNet
// (denoising_diffusion.py:92,98,114,200,222,225,253,254,297,339,354).
//
//   GEMM view:  M = output pixels (tile of 128 = R rows x Wt columns of ONE image),
//               N = output channels (tile BLOCK_N in {64,128,256}),
//               K = taps x input channels, consumed in blocks of 64 channels of one tap.
//
//   A operand:  activations are bf16 NHWC, i.e. every pixel is a 128-byte row per 64 channels.  A
//               K-block of A for tap (ky,kx) is the box {64 ch, Wt, R} of the input shifted by
//               (ky-pad, kx-pad): one TMA box load.  TMA zero-fills out-of-bounds elements, which
//               implements the convolution's zero padding with no branches and no im2col buffer;
//               the 128B-swizzled box lands in shared memory exactly in the canonical K-major
//               UMMA layout.  The skip-connection concat (:405,408,414) is a second tensor map
//               whose channels simply extend K; the pixel-unshuffle downsample (:95-99) is a 5-d
//               view (c, p2, w, p1, h) of the same tensor so its 1x1 conv needs no rearranged copy.
//   B operand:  weights packed bf16 [Cout][K] (K-major), 2-d TMA box {64, BLOCK_N}.
//   D:          fp32 in TMEM, double buffered (2 x BLOCK_N columns) so the epilogue of tile i
//               overlaps the MMAs of tile i+1.
//
//   Warp roles (192 threads, persistent CTA per SM, static round-robin tile schedule):
//     warp 0    TMA producer (one elected lane), STAGES-deep mbarrier ring
//     warp 1    TMEM allocator + MMA issuer (one lane issues tcgen05.mma, tcgen05.commit frees slots)
//     warps 2-5 epilogue: tcgen05.ld -> +bias (+residual) -> GroupNorm partial statistics
//               (sum, sum of squares per (sample, group), :176,181) -> bf16 NHWC store
#include "fd_conv_epi.cuh"

using namespace fdtc;

namespace {

constexpr int kBlockK = 64;
constexpr int kATileBytes = kBlockM * kBlockK * 2;  // 16 KiB
constexpr int kThreads = 64 + kEpiThreads + 32;     // warp 0 TMA (A), warp 1 MMA, warps 2..9 epilogue, warp 10 TMA (B)

struct ConvParams {
  int N, H, W;        // images, output rows, output columns (after flattening / merging)
  int Cout;
  int KW;             // taps per row
  int taps;           // KH*KW (4 for the pixel-unshuffle mode)
  int pad_h, pad_w;
  int mode;           // 0: conv taps with zero padding, 1: pixel-unshuffle + 1x1
  int chunks0, chunks1;  // 64-channel chunks of src0 / src1
  int R, Wt;          // tile = R rows x Wt columns, R*Wt == 128
  int tiles_w, tiles_h, n_tiles, total_tiles;
  const float* bias;
  const __nv_bfloat16* residual;
  double* gn_stats;   // [N][8][2] or null
  int shuffle_cq;     // > 0: pixel-shuffle store, out is (N, 2H, 2W, Cout/4)
  int dbg;            // FD_CONV_DBG in FD_DIAG builds (results are garbage): 1 = skip A loads, 2 = skip B loads, 4 = skip MMAs,
                      // 8 = skip the epilogue's work (barrier handshakes only)
  // residual transform (fd_conv_igemm_rt): `residual` is a raw conv output whose GroupNorm + SiLU the epilogue applies
  const double* rt_stats;
  const float* rt_gamma;
  const float* rt_beta;
  float rt_eps;
  int phase;          // >= 0: sub-pixel phase store (out_mode 2)
  // output head (fd_conv_igemm_rt_head): final 1x1 conv applied in the epilogue instead of storing the tile
  float* head_out;
  const float* head_w;
  const float* head_b;
  int head_n, head_h0, head_w0, head_pt, head_pl;
};

// SH ("store heavy"): few K-blocks per tile (1x1 convs), so the epilogue / output stores dominate: shallow operand
// ring, one staging slab per 64 output channels so no TMA store ever waits for a buffer.
template <int BLOCK_N, int SH = 0>
struct Cfg {
  static constexpr int kBTileBytes = BLOCK_N * kBlockK * 2;
  static constexpr int kStageBytes = kATileBytes + kBTileBytes;
  // SH: the tile is a pure stream (2-4 K-blocks, then 16-64 KB of output): the ring depth sets how many bytes an SM keeps in
  // flight against the DRAM latency -- 3 stages left the 128 -> 64 res_convs at 4.0 TB/s
  static constexpr int kStages = SH ? (BLOCK_N == 64 ? 6 : (BLOCK_N == 128 ? 5 : 3)) : (BLOCK_N == 64 ? 7 : (BLOCK_N == 128 ? 6 : 4));
  static constexpr int kStoreBufs = SH ? (BLOCK_N / 64 > 2 ? BLOCK_N / 64 : 2) : (BLOCK_N == 64 ? 2 : 1);   // staging slabs
  static constexpr int kTmemCols = 2 * BLOCK_N;
  static constexpr int kHeadBytes = BLOCK_N == 64 ? (256 + kEpiWarps * 32 * 4) * 4 : 0;      // output-head weights + exchange
  static constexpr int kTailBytes = 256 /*barriers*/ + 2 * BLOCK_N * 4 /*bias*/ + kEpiWarps * 16 * 4 /*stats*/ + 64 +
                                    4 * BLOCK_N * 4 /*residual-transform coefficients*/ + kHeadBytes;
  static constexpr int kSmemBytes = 1024 + kStages * kStageBytes + kStoreBufs * kSlabBytes + kTailBytes;
};

// GPT = GroupNorm groups covered by one N-tile (8 when Cout == BLOCK_N, 4 when Cout == 2*BLOCK_N, 0 = no statistics)
template <int BLOCK_N, int GPT, int SH>
__global__ void __launch_bounds__(kThreads, 1)
conv_igemm_kernel(const __grid_constant__ CUtensorMap map_a0, const __grid_constant__ CUtensorMap map_a1,
                  const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_out,
                  const ConvParams p) {
  using C = Cfg<BLOCK_N, SH>;
  constexpr int STAGES = C::kStages;
  constexpr int NBUF = C::kStoreBufs;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;   // SWIZZLE_128B tiles need 1024-byte alignment
  uint8_t* gbase = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t a_smem = base;
  const uint32_t b_smem = base + STAGES * kATileBytes;
  const uint32_t o_smem = base + STAGES * C::kStageBytes;
  const uint32_t bar_base = o_smem + NBUF * kSlabBytes;
  // barriers: full[STAGES], empty[STAGES], tmem_full[2], tmem_empty[2]
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + 2 + s); };
  uint8_t* gtail = gbase + STAGES * C::kStageBytes + NBUF * kSlabBytes + 256;
  float* s_bias = reinterpret_cast<float*>(gtail);                       // [2][BLOCK_N]
  float* s_stats = reinterpret_cast<float*>(gtail + 2 * BLOCK_N * 4);    // [8 warps][16]
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(gtail + 2 * BLOCK_N * 4 + kEpiWarps * 16 * 4);
  float* s_rt = reinterpret_cast<float*>(gtail + 2 * BLOCK_N * 4 + kEpiWarps * 16 * 4 + 64);        // [2][2][BLOCK_N]
  float* s_head = s_rt + 4 * BLOCK_N;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int cpt = p.chunks0 + p.chunks1;       // 64-channel chunks per tap
  const int num_kb = p.taps * cpt;
  const int tiles_per_img = p.tiles_w * p.tiles_h;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a0);
    tma_prefetch_desc(&map_a1);
    tma_prefetch_desc(&map_b);
    tma_prefetch_desc(&map_out);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 2);           // one arrive.expect_tx from each of the two producer threads
      mbar_init(empty_bar(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), kEpiThreads);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(s_tmem), C::kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;

  if (warp == 0 || warp == 10) {
    // ===================== TMA producers: warp 0 loads the activation tiles, warp 10 the weight tiles ==============
    // UTMALDG (like UTCHMMA below) takes its operands from uniform registers and releases them only when the TMA unit picks
    // the instruction up, i.e. when the previous box has been issued to memory: the first uniform-register write after a
    // cp.async.bulk.tensor stalls until then, and everything between that point and the next cp.async.bulk.tensor is time
    // the TMA unit sits idle.  Measured with FD_CONV_DBG on the N = 128 tiles: skipping the A loads 0.30 -> 0.19 ms, skipping
    // the B loads (short loop) nothing; every extra instruction in the A loop cost ~1 % of the kernel.  So all loop state is
    // made opaque to the uniform datapath (general registers), the coordinates are advanced incrementally (no division),
    // and only the register-to-uniform moves remain between two loads.
    if (elect_one_sync()) {
      int stage = opaque32(0);
      uint32_t phase = 0;
      const int tile0 = opaque32((int)blockIdx.x), tstep = opaque32((int)gridDim.x);
      if (warp == 0) {
        const bool skip = kDiag && (opaque32(p.dbg) & 1) != 0, mode0 = opaque32(p.mode) == 0;
        const int chunks0 = opaque32(p.chunks0), KW = opaque32(p.KW), cpt_ = opaque32(cpt), nkb = opaque32(num_kb);
        const uint64_t m0 = opaque64(reinterpret_cast<uint64_t>(&map_a0)), m1 = opaque64(reinterpret_cast<uint64_t>(&map_a1));
        for (int tile = tile0; tile < p.total_tiles; tile += tstep) {
          const int m_tile = tile / p.n_tiles;
          const int img = m_tile / tiles_per_img;
          const int rem = m_tile - img * tiles_per_img;
          const int th = rem / p.tiles_w;
          const int h0 = th * p.R;
          const int w0 = (rem - th * p.tiles_w) * p.Wt;
          // mode 0: (c, w0 + kx - pad, h0 + ky - pad, img, 0); mode 1: (c, kx, w0, ky, h0)
          const int bw = mode0 ? w0 - p.pad_w : 0, bh = mode0 ? h0 - p.pad_h : 0;
          int kx = 0, ky = 0, chunk = 0;
          for (int kb = 0; kb < nkb; ++kb) {
            // every operand of the load is final (and in a general register) BEFORE the barrier wait
            const bool first = chunk < chunks0;
            const uint64_t ma = opaque64(first ? m0 : m1);
            const int c0 = opaque32((first ? chunk : chunk - chunks0) * kBlockK);
            const int c1 = opaque32(bw + kx);
            const int c2 = opaque32(mode0 ? bh + ky : w0);
            const int c3 = opaque32(mode0 ? img : ky);
            const int c4 = opaque32(mode0 ? 0 : h0);
            const uint32_t fb = (uint32_t)opaque32((int)full_bar(stage));
            const uint32_t dst = (uint32_t)opaque32((int)(a_smem + stage * kATileBytes));
            mbar_wait(empty_bar(stage), phase ^ 1u);
            if (skip) {
              mbar_arrive(fb);
            } else {
              mbar_expect_tx(fb, kATileBytes);
              tma_load_5d(dst, reinterpret_cast<const CUtensorMap*>(ma), fb, c0, c1, c2, c3, c4);
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            if (++chunk == cpt_) {
              chunk = 0;
              if (++kx == KW) { kx = 0; ++ky; }
            }
          }
        }
      } else {
        const bool skip = kDiag && (opaque32(p.dbg) & 2) != 0;
        const int nkb = opaque32(num_kb);
        const uint64_t mb = opaque64(reinterpret_cast<uint64_t>(&map_b));
        for (int tile = tile0; tile < p.total_tiles; tile += tstep) {
          const int n0 = (tile % p.n_tiles) * BLOCK_N;
          int k0 = 0;
          for (int kb = 0; kb < nkb; ++kb, k0 += kBlockK) {
            const uint32_t fb = (uint32_t)opaque32((int)full_bar(stage));
            const uint32_t dst = (uint32_t)opaque32((int)(b_smem + stage * C::kBTileBytes));
            const int ck = opaque32(k0), cn = opaque32(n0);
            mbar_wait(empty_bar(stage), phase ^ 1u);
            if (skip) {
              mbar_arrive(fb);
            } else {
              mbar_expect_tx(fb, C::kBTileBytes);
              tma_load_2d(dst, reinterpret_cast<const CUtensorMap*>(mb), fb, ck, cn);
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (one elected lane runs the whole loop) =====================
    // UTCHMMA takes its descriptors from uniform registers and releases them only when the instruction is DISPATCHED to the
    // tensor pipe, i.e. when the previous MMA has finished: the first instruction after the four MMAs of a K-block that
    // overwrites a uniform register stalls until the fourth one starts executing, and whatever still has to run between that
    // point and the next K-block's first MMA (barrier wait, descriptor arithmetic) is exposed beyond the 64-128 cycles that
    // last MMA takes.  (Measured with FD_CONV_DBG: MMAs alone, no loads, no epilogue work: 525 cycles per N = 128 K-block =
    // 256 of MMA + ~255 of loop.)  So the loop is software-pipelined: the next K-block's barrier wait and descriptors (kept in
    // general registers, opaque to the uniform datapath) come BEFORE this K-block's commit, and only register-to-uniform moves
    // are left on the exposed path.
    constexpr uint32_t idesc = umma_idesc_bf16(kBlockM, BLOCK_N);
    if (elect_one_sync()) {
      const uint64_t adesc0 = umma_desc_sw128(a_smem), bdesc0 = umma_desc_sw128(b_smem);
      int stage = 0;
      uint32_t phase = 0;
      int iter = 0;
      bool waited = false;
      const bool skip_mma = kDiag && (p.dbg & 4) != 0;
      uint64_t ad = opaque64(adesc0), bd = opaque64(bdesc0);
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++iter) {
        const int as = iter & 1;
        const uint32_t aphase = (iter >> 1) & 1;
        mbar_wait(tempty_bar(as), aphase ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * BLOCK_N;
        for (int kb = 0; kb < num_kb; ++kb) {
          if (!waited) mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          if (!skip_mma) {
#pragma unroll
            for (int k = 0; k < kBlockK / 16; ++k) {
              // advance 16 bf16 (32 B) along K inside the 128-byte swizzle atom: +2 in the (addr >> 4) field
              umma_bf16(tmem_d, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
            }
          }
          const uint32_t cur_empty = empty_bar(stage);
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          ad = opaque64(adesc0 + (uint64_t)(stage * (kATileBytes >> 4)));
          bd = opaque64(bdesc0 + (uint64_t)(stage * (C::kBTileBytes >> 4)));
          waited = kb + 1 < num_kb;
          if (waited) mbar_wait(full_bar(stage), phase);
          umma_commit(cur_empty);                             // frees the smem slot when the MMAs retire
          if (kb == num_kb - 1) umma_commit(tfull_bar(as));   // accumulator complete -> epilogue
        }
      }
    }
    __syncwarp();
  } else if (warp >= 2 && warp < 2 + kEpiWarps) {
    // ===================== epilogue (warps 2..9) =====================
    EpiCtx ec;
    ec.tmem_base = tmem_base;
    ec.o_smem = o_smem;
    ec.tfull0 = tfull_bar(0);
    ec.tempty0 = tempty_bar(0);
    ec.s_bias = s_bias;
    ec.s_stats = s_stats;
    ec.map_out = &map_out;
    ec.bias = p.bias;
    ec.residual = p.residual;
    ec.gn_stats = p.gn_stats;
    ec.H = p.H; ec.W = p.W; ec.Cout = p.Cout; ec.Wt = p.Wt;
    ec.shuffle_cq = p.shuffle_cq;
    ec.tempty_remote = 0;
    ec.dbg = kDiag ? p.dbg : 0;
    ec.rt_stats = p.rt_stats; ec.rt_gamma = p.rt_gamma; ec.rt_beta = p.rt_beta; ec.rt_eps = p.rt_eps; ec.s_rt = s_rt;
    ec.phase = p.phase;
    ec.head_out = p.head_out; ec.head_w = p.head_w; ec.head_b = p.head_b; ec.head_n = p.head_n; ec.s_head = s_head;
    ec.head_h0 = p.head_h0; ec.head_w0 = p.head_w0; ec.head_pt = p.head_pt; ec.head_pl = p.head_pl;
    conv_epilogue<BLOCK_N, GPT, NBUF>(ec, [&](int iter, EpiTile& t) {
      const int tile = blockIdx.x + iter * gridDim.x;
      if (tile >= p.total_tiles) return false;
      t.n_tile = tile % p.n_tiles;
      const int m_tile = tile / p.n_tiles;
      t.img = m_tile / tiles_per_img;
      const int rem = m_tile - t.img * tiles_per_img;
      t.h0 = (rem / p.tiles_w) * p.R;
      t.w0 = (rem % p.tiles_w) * p.Wt;
      return true;
    });
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------
// CTA-pair variant for the N = 128 / 256 tiles (Cout % 128 == 0): cta_group::2, M = 256 = two 128-pixel tiles.
// Measured (scripts/micro/umma_rate*.cu, profiles/r1_umma_rate.txt): a single CTA moves fill + operand reads of
// 48 + 48 KB per 512 tensor cycles through its 128 B/clk shared-memory pipe (187 B/clk needed -> ~67 % of peak); in a
// pair each CTA fills and holds only HALF of the weight tile, which the hardware shares: 32 + 32 KB = 125 B/clk.
//   * both CTAs run a TMA producer: own activation tile + own half (128 rows) of the weight tile, all transaction bytes
//     signalled on the LEADER's full barrier (cp.async.bulk.tensor ... cta_group::2, barrier address with the peer bit
//     cleared);
//   * only the leader issues tcgen05.mma.cta_group::2 (idesc M = 256); tcgen05.commit ... multicast::cluster frees the
//     stage / publishes the accumulator in BOTH CTAs;
//   * each CTA's epilogue drains its own 128 TMEM lanes; the non-leader's "drained" arrivals go to the leader's barrier.
// ------------------------------------------------------------------------------------------------
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma2_load_5d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2, int c3,
                                             int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(dst),
      "l"(m), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma2_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(m), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma2_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}

// MT = M-tiles (128 pixels each) per CTA and K-block.  MT = 2 (N = 128 only): the pair works on FOUR M-tiles that share one
// weight tile, so a K-block moves 32 KB of activations + 8 KB of weights per CTA for eight 64-cycle MMAs = 80 B/clk instead
// of 96 -- the N = 128 tiles are bound by the L2 -> SM delivery rate (~74 B/clk/SM measured, profiles/r1_conv_diag_n128.txt).
template <int BLOCK_N, int MT = 1>
struct PairCfg {
  static constexpr int kBHalfBytes = (BLOCK_N / 2) * kBlockK * 2;   // this CTA's half of the weight tile's rows
  static constexpr int kStageBytes = MT * kATileBytes + kBHalfBytes;     // 32 / 24 / 40 KiB
  static constexpr int kStages = MT == 2 ? 5 : (BLOCK_N == 256 ? 5 : 7);
  static constexpr int kStoreBufs = MT == 2 ? 1 : 2;             // MT = 2: the fifth ring stage is worth more than a second slab
  static constexpr int kAcc = 2 * MT;                               // accumulator stages
  static constexpr int kTmemCols = kAcc * BLOCK_N;
  static constexpr int kTailBytes = 256 + 2 * BLOCK_N * 4 + kEpiWarps * 16 * 4 + 64 + 4 * BLOCK_N * 4;
  static constexpr int kSmemBytes = 1024 + kStages * kStageBytes + kStoreBufs * kSlabBytes + kTailBytes;
  static_assert(kTmemCols <= 512, "accumulators do not fit tensor memory");
};

template <int BLOCK_N, int GPT, int MT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
conv_igemm_pair_kernel(const __grid_constant__ CUtensorMap map_a0, const __grid_constant__ CUtensorMap map_a1,
                       const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_out,
                       const ConvParams p) {
  using C = PairCfg<BLOCK_N, MT>;
  constexpr int STAGES = C::kStages;
  constexpr int NBUF = C::kStoreBufs;
  constexpr int NACC = C::kAcc;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t a_smem = base;
  const uint32_t b_smem = base + STAGES * MT * kATileBytes;
  const uint32_t o_smem = base + STAGES * C::kStageBytes;
  const uint32_t bar_base = o_smem + NBUF * kSlabBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + NACC + s); };
  uint8_t* gtail = gbase + STAGES * C::kStageBytes + NBUF * kSlabBytes + 256;
  float* s_bias = reinterpret_cast<float*>(gtail);
  float* s_stats = reinterpret_cast<float*>(gtail + 2 * BLOCK_N * 4);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(gtail + 2 * BLOCK_N * 4 + kEpiWarps * 16 * 4);
  float* s_rt = reinterpret_cast<float*>(gtail + 2 * BLOCK_N * 4 + kEpiWarps * 16 * 4 + 64);        // [2][2][BLOCK_N]
  float* s_head = nullptr;      // (the output head is an N = 64, single-CTA feature)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int cpt = p.chunks0 + p.chunks1;
  const int num_kb = p.taps * cpt;
  const int tiles_per_img = p.tiles_w * p.tiles_h;
  const int super_tiles = p.total_tiles / (2 * MT);     // (2 MT M-tiles) x N-tile; the host guarantees the M count divides

  auto decode = [&](int st, int m, int& n_tile, int& img, int& h0, int& w0) {
    n_tile = st % p.n_tiles;
    const int m_tile = 2 * MT * (st / p.n_tiles) + (int)rank * MT + m;
    img = m_tile / tiles_per_img;
    const int rem = m_tile - img * tiles_per_img;
    h0 = (rem / p.tiles_w) * p.R;
    w0 = (rem % p.tiles_w) * p.Wt;
  };

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a0);
    tma_prefetch_desc(&map_a1);
    tma_prefetch_desc(&map_b);
    tma_prefetch_desc(&map_out);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 2);                       // the leader's two producer threads (expect_tx for both CTAs' bytes)
      mbar_init(empty_bar(s), 1);
    }
    for (int s = 0; s < NACC; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), 2 * kEpiThreads);       // both CTAs' epilogues arrive on the leader's barrier
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(C::kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                   // peers' barriers are initialised before anyone signals them
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;

  if (warp == 0 || warp == 10) {
    // ===================== TMA producers (both CTAs): warp 0 activation tiles, warp 10 weight half-tiles ==========
    // (loop structure: see conv_igemm_kernel -- every operand final and in a general register before the barrier wait)
    if (elect_one_sync()) {
      int stage = opaque32(0);
      uint32_t phase = 0;
      const int st0 = opaque32(pair), ststep = opaque32(npairs), nkb = opaque32(num_kb);
      const bool leader = opaque32((int)rank) == 0;
      if (warp == 0) {
        const bool mode0 = opaque32(p.mode) == 0;
        const int chunks0 = opaque32(p.chunks0), KW = opaque32(p.KW), cpt_ = opaque32(cpt);
        const uint64_t m0 = opaque64(reinterpret_cast<uint64_t>(&map_a0)), m1 = opaque64(reinterpret_cast<uint64_t>(&map_a1));
        for (int st = st0; st < super_tiles; st += ststep) {
          int n_tile, img[MT], h0[MT], w0[MT], bw[MT], bh[MT];
#pragma unroll
          for (int m = 0; m < MT; ++m) {
            decode(st, m, n_tile, img[m], h0[m], w0[m]);
            bw[m] = mode0 ? w0[m] - p.pad_w : 0;
            bh[m] = mode0 ? h0[m] - p.pad_h : 0;
          }
          int kx = 0, ky = 0, chunk = 0;
          for (int kb = 0; kb < nkb; ++kb) {
            const bool first = chunk < chunks0;
            const uint64_t ma = opaque64(first ? m0 : m1);
            const int c0 = opaque32((first ? chunk : chunk - chunks0) * kBlockK);
            int c1[MT], c2[MT], c3[MT], c4[MT];
#pragma unroll
            for (int m = 0; m < MT; ++m) {
              c1[m] = opaque32(bw[m] + kx);
              c2[m] = opaque32(mode0 ? bh[m] + ky : w0[m]);
              c3[m] = opaque32(mode0 ? img[m] : ky);
              c4[m] = opaque32(mode0 ? 0 : h0[m]);
            }
            const uint32_t fb = (uint32_t)opaque32((int)full_bar(stage));
            const uint32_t dst = (uint32_t)opaque32((int)(a_smem + stage * MT * kATileBytes));
            mbar_wait(empty_bar(stage), phase ^ 1u);
            if (kDiag && (p.dbg & 1)) {
              if (leader) mbar_arrive(fb);
            } else {
              if (leader) mbar_expect_tx(fb, 2 * MT * kATileBytes);                   // both CTAs' activation tiles
#pragma unroll
              for (int m = 0; m < MT; ++m)
                tma2_load_5d(dst + m * kATileBytes, reinterpret_cast<const CUtensorMap*>(ma), fb, c0, c1[m], c2[m], c3[m], c4[m]);
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            if (++chunk == cpt_) {
              chunk = 0;
              if (++kx == KW) { kx = 0; ++ky; }
            }
          }
        }
      } else {
        const uint64_t mb = opaque64(reinterpret_cast<uint64_t>(&map_b));
        for (int st = st0; st < super_tiles; st += ststep) {
          const int n0 = (st % p.n_tiles) * BLOCK_N + (int)rank * (BLOCK_N / 2);
          int k0 = 0;
          for (int kb = 0; kb < nkb; ++kb, k0 += kBlockK) {
            const uint32_t fb = (uint32_t)opaque32((int)full_bar(stage));
            const uint32_t dst = (uint32_t)opaque32((int)(b_smem + stage * C::kBHalfBytes));
            const int ck = opaque32(k0), cn = opaque32(n0);
            mbar_wait(empty_bar(stage), phase ^ 1u);
            if (kDiag && (p.dbg & 2)) {
              if (leader) mbar_arrive(fb);
            } else {
              if (leader) mbar_expect_tx(fb, 2 * C::kBHalfBytes);                    // both CTAs' halves of the weight tile
              tma2_load_2d(dst, reinterpret_cast<const CUtensorMap*>(mb), fb, ck, cn);
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only; software-pipelined like conv_igemm_kernel's) ==============
    if (rank == 0 && elect_one_sync()) {
      constexpr uint32_t idesc = umma_idesc_bf16(256, BLOCK_N);
      const uint64_t adesc0 = umma_desc_sw128(a_smem), bdesc0 = umma_desc_sw128(b_smem);
      int stage = 0;
      uint32_t phase = 0;
      int iter = 0;
      bool waited = false;
      uint64_t ad = opaque64(adesc0), bd = opaque64(bdesc0);
      for (int st = pair; st < super_tiles; st += npairs, ++iter) {
        const int as0 = (iter & 1) * MT;                      // this super-tile's first accumulator stage
        const uint32_t aphase = (iter >> 1) & 1;
#pragma unroll
        for (int m = 0; m < MT; ++m) mbar_wait(tempty_bar(as0 + m), aphase ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as0 * BLOCK_N;
        for (int kb = 0; kb < num_kb; ++kb) {
          if (!waited) mbar_wait(full_bar(stage), phase);
          tc_fence_after();
#pragma unroll
          for (int m = 0; m < MT; ++m)
#pragma unroll
            for (int k = 0; k < kBlockK / 16; ++k)
              if (!(kDiag && (p.dbg & 4)))
                umma2_bf16(tmem_d + m * BLOCK_N, ad + (uint64_t)(m * (kATileBytes >> 4) + 2 * k), bd + (uint64_t)(2 * k), idesc,
                           (kb | k) != 0 ? 1u : 0u);
          const uint32_t cur_empty = empty_bar(stage);
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          ad = opaque64(adesc0 + (uint64_t)(stage * (MT * kATileBytes >> 4)));
          bd = opaque64(bdesc0 + (uint64_t)(stage * (C::kBHalfBytes >> 4)));
          waited = kb + 1 < num_kb;
          if (waited) mbar_wait(full_bar(stage), phase);
          umma2_commit(cur_empty);
          if (kb == num_kb - 1) {
#pragma unroll
            for (int m = 0; m < MT; ++m) umma2_commit(tfull_bar(as0 + m));
          }
        }
      }
    }
    __syncwarp();
  } else if (warp >= 2 && warp < 2 + kEpiWarps) {
    // ===================== epilogue (warps 2..9 of both CTAs): own 128 TMEM lanes =====================
    EpiCtx ec;
    ec.tmem_base = tmem_base;
    ec.o_smem = o_smem;
    ec.tfull0 = tfull_bar(0);
    ec.tempty0 = tempty_bar(0);
    ec.s_bias = s_bias;
    ec.s_stats = s_stats;
    ec.map_out = &map_out;
    ec.bias = p.bias;
    ec.residual = p.residual;
    ec.gn_stats = p.gn_stats;
    ec.H = p.H; ec.W = p.W; ec.Cout = p.Cout; ec.Wt = p.Wt;
    ec.shuffle_cq = p.shuffle_cq;
    ec.tempty_remote = rank != 0;
    ec.dbg = kDiag ? p.dbg : 0;
    ec.rt_stats = p.rt_stats; ec.rt_gamma = p.rt_gamma; ec.rt_beta = p.rt_beta; ec.rt_eps = p.rt_eps; ec.s_rt = s_rt;
    ec.phase = p.phase;
    ec.head_out = p.head_out; ec.head_w = p.head_w; ec.head_b = p.head_b; ec.head_n = p.head_n; ec.s_head = s_head;
    ec.head_h0 = p.head_h0; ec.head_w0 = p.head_w0; ec.head_pt = p.head_pt; ec.head_pl = p.head_pl;
    conv_epilogue<BLOCK_N, GPT, NBUF, NACC>(ec, [&](int iter, EpiTile& t) {
      const int st = pair + (iter / MT) * npairs;
      if (st >= super_tiles) return false;
      decode(st, iter % MT, t.n_tile, t.img, t.h0, t.w0);
      return true;
    });
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                   // nobody exits while the peer may still touch its barriers / smem
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(C::kTmemCols) : "memory");
  }
}

template <int BLOCK_N, int GPT, int MT = 1>
int launch_pair(const CUtensorMap& ma0, const CUtensorMap& ma1, const CUtensorMap& mb, const CUtensorMap& mo, const ConvParams& p,
                int sms, cudaStream_t st) {
  using C = PairCfg<BLOCK_N, MT>;
  static bool attr_set = false;
  if (!attr_set) {
    FD_CUDA(cudaFuncSetAttribute(conv_igemm_pair_kernel<BLOCK_N, GPT, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 C::kSmemBytes));
    attr_set = true;
  }
  const int units = p.total_tiles / MT;                  // CTA-sized work units
  int grid = units < sms ? units : sms;
  grid &= ~1;
  conv_igemm_pair_kernel<BLOCK_N, GPT, MT><<<grid, kThreads, C::kSmemBytes, st>>>(ma0, ma1, mb, mo, p);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

struct TileShape {
  int R, Wt;
};

// R x Wt = 128 covering an H x W image with the least padding waste (ties -> widest tile)
TileShape pick_tile(int H, int W) {
  TileShape best{1, 128};
  long best_cost = -1;
  for (int wt = 128; wt >= 8; wt >>= 1) {
    const int r = 128 / wt;
    const long cost = (long)((W + wt - 1) / wt) * wt * (long)((H + r - 1) / r) * r;
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best = TileShape{r, wt};
    }
  }
  return best;
}

// the same restricted to R | H: the phase store (out_mode 2) addresses rows of all images as one dimension, so a tile must not
// overhang the bottom of its image (the TMA store could not clip it)
TileShape pick_tile_rows_divide(int H, int W) {
  TileShape best{1, 128};
  long best_cost = -1;
  for (int wt = 128; wt >= 8; wt >>= 1) {
    const int r = 128 / wt;
    if (H % r != 0) continue;
    const long cost = (long)((W + wt - 1) / wt) * wt * (long)H;
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best = TileShape{r, wt};
    }
  }
  return best;
}

template <int BLOCK_N, int GPT, int SH = 0>
int launch(const CUtensorMap& ma0, const CUtensorMap& ma1, const CUtensorMap& mb, const CUtensorMap& mo,
           const ConvParams& p, int sms, cudaStream_t st) {
  using C = Cfg<BLOCK_N, SH>;
  static bool attr_set = false;
  if (!attr_set) {
    FD_CUDA(cudaFuncSetAttribute(conv_igemm_kernel<BLOCK_N, GPT, SH>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 C::kSmemBytes));
    attr_set = true;
  }
  const int grid = p.total_tiles < sms ? p.total_tiles : sms;
  conv_igemm_kernel<BLOCK_N, GPT, SH><<<grid, kThreads, C::kSmemBytes, st>>>(ma0, ma1, mb, mo, p);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

}  // namespace

int fd_conv3x3_strip_launch(const void* src0, int C0, const void* src1, int C1, const void* wpacked, const float* bias,
                            const void* residual,
                            void* out, double* gn_stats, int N, int H, int W, cudaStream_t st);   // fd_conv_strip.cu

struct HeadArgs {           // fd_conv_igemm_rt_head: see EpiCtx::head_*
  float* out;
  const float* w;
  const float* b;
  int n, h0, w0, pt, pl;
};

static int conv_igemm_impl(const void* src0, int C0, const void* src1, int C1, const void* wpacked, const float* bias,
                           const void* residual, void* out, double* gn_stats, int N, int H, int W, int Cout, int KH, int KW,
                           int pad_h, int pad_w, int mode, int out_mode, const double* rt_stats, const float* rt_gamma,
                           const float* rt_beta, float rt_eps, void* stream, int phase = -1, const struct HeadArgs* head = nullptr);

extern "C" {

int fd_conv_igemm(const void* src0, int C0, const void* src1, int C1, const void* wpacked, const float* bias,
                  const void* residual, void* out, double* gn_stats, int N, int H, int W, int Cout, int KH, int KW,
                  int pad_h, int pad_w, int mode, void* stream) {
  return fd_conv_igemm_ex(src0, C0, src1, C1, wpacked, bias, residual, out, gn_stats, N, H, W, Cout, KH, KW, pad_h,
                          pad_w, mode, 0, stream);
}

int fd_conv_igemm_ex(const void* src0, int C0, const void* src1, int C1, const void* wpacked, const float* bias,
                     const void* residual, void* out, double* gn_stats, int N, int H, int W, int Cout, int KH, int KW,
                     int pad_h, int pad_w, int mode, int out_mode, void* stream) {
  return conv_igemm_impl(src0, C0, src1, C1, wpacked, bias, residual, out, gn_stats, N, H, W, Cout, KH, KW, pad_h, pad_w, mode,
                         out_mode, nullptr, nullptr, nullptr, 0.f, stream);
}

int fd_conv_igemm_rt(const void* src0, int C0, const void* src1, int C1, const void* wpacked, const float* bias,
                     const void* residual_raw, const double* res_stats, const float* res_gamma, const float* res_beta, float eps,
                     void* out, int N, int H, int W, int Cout, int KH, int KW, int pad_h, int pad_w, void* stream) {
  FD_REQUIRE(residual_raw && res_stats && res_gamma && res_beta, "conv_igemm_rt: null pointer");
  FD_REQUIRE(Cout % 64 == 0 && (Cout / 8) > 0, "conv_igemm_rt: Cout=%d", Cout);
  return conv_igemm_impl(src0, C0, src1, C1, wpacked, bias, residual_raw, out, nullptr, N, H, W, Cout, KH, KW, pad_h, pad_w, 0, 0,
                         res_stats, res_gamma, res_beta, eps, stream);
}

int fd_conv_igemm_rt_head(const void* src0, int C0, const void* src1, int C1, const void* wpacked, const float* bias,
                          const void* residual_raw, const double* res_stats, const float* res_gamma, const float* res_beta, float eps,
                          const float* head_w, const float* head_b, int head_n, float* out_nchw, int N, int H, int W, int H0, int W0,
                          int pad_top, int pad_left, void* stream) {
  FD_REQUIRE(residual_raw && res_stats && res_gamma && res_beta && head_w && head_b && out_nchw, "conv_igemm_rt_head: null pointer");
  FD_REQUIRE(head_n >= 1 && head_n <= 4, "conv_igemm_rt_head: head_n=%d (1..4)", head_n);
  FD_REQUIRE(H0 > 0 && W0 > 0 && pad_top >= 0 && pad_left >= 0 && pad_top + H0 <= H && pad_left + W0 <= W,
             "conv_igemm_rt_head: crop %dx%d at (%d, %d) outside %dx%d", H0, W0, pad_top, pad_left, H, W);
  const HeadArgs ha{out_nchw, head_w, head_b, head_n, H0, W0, pad_top, pad_left};
  return conv_igemm_impl(src0, C0, src1, C1, wpacked, bias, residual_raw, nullptr, nullptr, N, H, W, 64, 1, 1, 0, 0, 0, 0,
                         res_stats, res_gamma, res_beta, eps, stream, -1, &ha);
}

int fd_conv_igemm_up(const void* src, int Cin, const void* wpacked4, const float* bias, void* out, int N, int H, int W, int Cout,
                     void* stream) {
  FD_REQUIRE(src && wpacked4 && out, "conv_igemm_up: null pointer");
  FD_REQUIRE(Cin % 64 == 0 && Cout % 64 == 0, "conv_igemm_up: Cin=%d Cout=%d must be multiples of 64", Cin, Cout);
  const __nv_bfloat16* w4 = static_cast<const __nv_bfloat16*>(wpacked4);
  for (int ph = 0; ph < 4; ++ph) {
    // phase (a, b): 2x2 taps on the low-resolution grid, tap (ty, tx) reads (i + ty - (1 - a), j + tx - (1 - b))
    const int a = ph >> 1, b = ph & 1;
    if (int e = conv_igemm_impl(src, Cin, nullptr, 0, w4 + (size_t)ph * Cout * 4 * Cin, bias, nullptr, out, nullptr, N, H, W, Cout, 2, 2,
                                1 - a, 1 - b, 0, 2, nullptr, nullptr, nullptr, 0.f, stream, ph))
      return e;
  }
  return FD_OK;
}

}  // extern "C"

static int conv_igemm_impl(const void* src0, int C0, const void* src1, int C1, const void* wpacked, const float* bias,
                           const void* residual, void* out, double* gn_stats, int N, int H, int W, int Cout, int KH, int KW,
                           int pad_h, int pad_w, int mode, int out_mode, const double* rt_stats, const float* rt_gamma,
                           const float* rt_beta, float rt_eps, void* stream, int phase, const HeadArgs* head) {
  FD_REQUIRE(head == nullptr || (Cout == 64 && rt_stats != nullptr && out_mode == 0 && mode == 0 && gn_stats == nullptr && KH == 1 && KW == 1),
             "conv_igemm: the output head takes a 1x1 residual-transform conv with Cout = 64");
  if (head != nullptr && out == nullptr) out = const_cast<void*>(src0);      // (tensor map only; the head never stores the tile)
  FD_REQUIRE(out_mode == 0 || out_mode == 1 || out_mode == 2, "conv_igemm: out_mode %d", out_mode);
  FD_REQUIRE(out_mode != 2 || (mode == 0 && phase >= 0 && phase < 4 && residual == nullptr && gn_stats == nullptr && rt_stats == nullptr),
             "conv_igemm: the phase store takes a plain conv (no residual / statistics)");
  FD_REQUIRE(out_mode != 1 || (mode == 0 && KH == 1 && KW == 1 && pad_h == 0 && pad_w == 0 && C1 == 0 &&
                               residual == nullptr && gn_stats == nullptr && Cout % 256 == 0),
             "conv_igemm: the pixel-shuffle store is for 1x1 convs with Cout %% 256 == 0, no residual / statistics");
  FD_REQUIRE(src0 && wpacked && out, "conv_igemm: null pointer");
  FD_REQUIRE(N > 0 && H > 0 && W > 0, "conv_igemm: bad geometry N=%d H=%d W=%d", N, H, W);
  FD_REQUIRE(C0 > 0 && C0 % 64 == 0 && C1 >= 0 && C1 % 64 == 0, "conv_igemm: C0=%d C1=%d must be multiples of 64", C0, C1);
  FD_REQUIRE(src1 != nullptr || C1 == 0, "conv_igemm: C1 > 0 needs src1");
  FD_REQUIRE(Cout > 0 && Cout % 64 == 0, "conv_igemm: Cout=%d must be a multiple of 64", Cout);
  FD_REQUIRE(mode == 0 || mode == 1, "conv_igemm: mode %d", mode);
  FD_REQUIRE(mode == 0 || (C1 == 0 && gn_stats == nullptr), "conv_igemm: mode 1 takes one source and no statistics");
  FD_REQUIRE(KH >= 1 && KW >= 1 && KH * KW <= 64, "conv_igemm: bad kernel %dx%d", KH, KW);
  {
    // large-image {64,128} -> 64 3x3 layers: rolling-strip kernel (each input pixel is fetched from L2 once
    // instead of nine times; the 64 -> 64 weights stay resident in shared memory)
    const bool chans_ok = (C0 == 64 && (C1 == 0 || C1 == 64)) || (C0 == 128 && C1 == 0);
    if (mode == 0 && KH == 3 && KW == 3 && pad_h == 1 && pad_w == 1 && chans_ok && Cout == 64 && W >= 128 && out_mode == 0 &&
        rt_stats == nullptr)
      return fd_conv3x3_strip_launch(src0, C0, src1, C1, wpacked, bias, residual, out, gn_stats, N, H, W, (cudaStream_t)stream);
  }
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    FD_CUDA(cudaGetDevice(&dev));
    FD_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  }
  ConvParams p{};
  p.Cout = Cout;
  p.mode = mode;
  p.chunks0 = C0 / 64;
  p.chunks1 = C1 / 64;
  p.bias = bias;
  p.residual = static_cast<const __nv_bfloat16*>(residual);
  p.gn_stats = gn_stats;
  p.rt_stats = rt_stats; p.rt_gamma = rt_gamma; p.rt_beta = rt_beta; p.rt_eps = rt_eps;
  p.phase = out_mode == 2 ? phase : -1;
  if (head != nullptr) {
    p.head_out = head->out; p.head_w = head->w; p.head_b = head->b; p.head_n = head->n;
    p.head_h0 = head->h0; p.head_w0 = head->w0; p.head_pt = head->pt; p.head_pl = head->pl;
  }
  CUtensorMap ma0, ma1, mb, mo;
  TileShape ts;
  if (mode == 0) {
    int n = N, h = H, w = W;
    if (out_mode == 1) {
      // no halo: rows of all images merge; the real (h, w) geometry is kept for the shuffled store
      n = 1;
      h = N * H;
    } else if (KH == 1 && KW == 1 && pad_h == 0 && pad_w == 0 && gn_stats == nullptr && rt_stats == nullptr) {
      // 1x1: no halo, so every pixel of the batch is one long row -> full 128-pixel tiles for any W
      FD_REQUIRE((long)N * H * W < (1L << 31), "conv_igemm: too many pixels");
      w = N * H * W;
      h = 1;
      n = 1;
    }
    p.N = n; p.H = h; p.W = w;
    p.KW = KW;
    p.taps = KH * KW;
    p.pad_h = pad_h;
    p.pad_w = pad_w;
    ts = out_mode == 2 ? pick_tile_rows_divide(h, w) : pick_tile(h, w);
    const uint32_t box[5] = {64, (uint32_t)ts.Wt, (uint32_t)ts.R, 1, 1};
    {
      const uint64_t dims[5] = {(uint64_t)C0, (uint64_t)w, (uint64_t)h, (uint64_t)n, 1};
      const uint64_t str[4] = {(uint64_t)C0 * 2, (uint64_t)w * C0 * 2, (uint64_t)h * w * C0 * 2, (uint64_t)n * h * w * C0 * 2};
      if (int e = make_tmap_bf16(&ma0, src0, 5, dims, str, box)) return e;
    }
    if (C1 > 0) {
      const uint64_t dims[5] = {(uint64_t)C1, (uint64_t)w, (uint64_t)h, (uint64_t)n, 1};
      const uint64_t str[4] = {(uint64_t)C1 * 2, (uint64_t)w * C1 * 2, (uint64_t)h * w * C1 * 2, (uint64_t)n * h * w * C1 * 2};
      if (int e = make_tmap_bf16(&ma1, src1, 5, dims, str, box)) return e;
    } else {
      ma1 = ma0;
    }
  } else {
    // src is (N, 2H, 2W, C0); output rows of all images are merged (no halo -> tiles may span images)
    p.N = 1; p.H = N * H; p.W = W;
    p.KW = 2;
    p.taps = 4;
    ts = pick_tile(p.H, p.W);
    const uint64_t dims[5] = {(uint64_t)C0, 2, (uint64_t)W, 2, (uint64_t)N * H};
    const uint64_t str[4] = {(uint64_t)C0 * 2, (uint64_t)2 * C0 * 2, (uint64_t)2 * W * C0 * 2, (uint64_t)4 * W * C0 * 2};
    const uint32_t box[5] = {64, 1, (uint32_t)ts.Wt, 1, (uint32_t)ts.R};
    if (int e = make_tmap_bf16(&ma0, src0, 5, dims, str, box)) return e;
    ma1 = ma0;
  }
  p.R = ts.R;
  p.Wt = ts.Wt;
  p.tiles_w = (p.W + ts.Wt - 1) / ts.Wt;
  p.tiles_h = (p.H + ts.R - 1) / ts.R;
  const int block_n = (Cout % 256 == 0) ? 256 : ((Cout % 128 == 0) ? 128 : 64);
  p.n_tiles = Cout / block_n;
  const long total = (long)p.N * p.tiles_w * p.tiles_h * p.n_tiles;
  FD_REQUIRE(total < (1L << 31), "conv_igemm: too many tiles");
  p.total_tiles = (int)total;
  const bool stats_ = gn_stats != nullptr;
  const bool store_heavy_ = !stats_ && p.taps * (p.chunks0 + p.chunks1) <= 4;
  // CTA pairs (cta_group::2): needs an even number of M-tiles (two per pair).  Measured at batch 8, 440x1024 shapes
  // (after the elect.sync fix removed the single-thread issue overhead, which had made the leader the bottleneck):
  // N = 256 tiles +2 % (those layers already run at the power-limited practical peak, cuBLAS burst = 1.65 PF/s);
  // N = 128 tiles 0.97-0.99 PF/s vs 0.93-0.96 single (+3-4 %: each CTA stages only half of B, so the TMA fill traffic
  // per MMA drops).  Both widths therefore run as pairs.
  static const int dbg = fd_diag_bits("FD_CONV_DBG");
  p.dbg = dbg;
  const bool use_pair = block_n >= 128 && !store_heavy_ && out_mode != 1 && ((long)p.N * p.tiles_w * p.tiles_h) % 2 == 0 &&
                        p.total_tiles >= 2;
  {
    const uint64_t K = (uint64_t)p.taps * (C0 + C1);
    const uint64_t dims[2] = {K, (uint64_t)Cout};
    const uint64_t str[1] = {K * 2};
    const uint32_t box[2] = {64, (uint32_t)(use_pair ? block_n / 2 : block_n)};
    if (int e = make_tmap_bf16(&mb, wpacked, 2, dims, str, box)) return e;
  }
  if (out_mode == 1) {
    // dgrad of Downsample (:95-99): channel (p1*2+p2)*Cq + c of pixel (h, w) goes to pixel (2h+p1, 2w+p2), channel c
    const uint64_t cq = (uint64_t)Cout / 4;
    p.shuffle_cq = (int)cq;
    const uint64_t dims[5] = {cq, 2, (uint64_t)p.W, 2, (uint64_t)p.H};
    const uint64_t str[4] = {cq * 2, 2 * cq * 2, (uint64_t)2 * p.W * cq * 2, (uint64_t)4 * p.W * cq * 2};
    const uint32_t box[5] = {64, 1, (uint32_t)ts.Wt, 1, (uint32_t)ts.R};
    if (int e = make_tmap_bf16(&mo, out, 5, dims, str, box)) return e;
  } else if (out_mode == 2) {
    // sub-pixel phase store: out is (N, 2H, 2W, Cout); the tile of low-resolution pixels (h, w) goes to (2h + a, 2w + b)
    const uint64_t c = (uint64_t)Cout;
    const uint64_t dims[5] = {c, 2, (uint64_t)p.W, 2, (uint64_t)p.N * p.H};
    const uint64_t str[4] = {c * 2, 2 * c * 2, (uint64_t)2 * p.W * c * 2, (uint64_t)4 * p.W * c * 2};
    const uint32_t box[5] = {64, 1, (uint32_t)ts.Wt, 1, (uint32_t)ts.R};
    if (int e = make_tmap_bf16(&mo, out, 5, dims, str, box)) return e;
  } else {
    // output (N, H, W, Cout) in the same (possibly flattened / merged) geometry: box = one 64-channel slab of a tile
    const uint64_t dims[5] = {(uint64_t)Cout, (uint64_t)p.W, (uint64_t)p.H, (uint64_t)p.N, 1};
    const uint64_t str[4] = {(uint64_t)Cout * 2, (uint64_t)p.W * Cout * 2, (uint64_t)p.H * p.W * Cout * 2,
                             (uint64_t)p.N * p.H * p.W * Cout * 2};
    const uint32_t box[5] = {64, (uint32_t)ts.Wt, (uint32_t)ts.R, 1, 1};
    if (int e = make_tmap_bf16(&mo, out, 5, dims, str, box)) return e;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const bool stats = gn_stats != nullptr;
  if (stats) FD_REQUIRE(p.n_tiles == 1 || p.n_tiles == 2, "conv_igemm: statistics need Cout in {64,128,256,512}");
  const bool store_heavy = !stats && p.taps * (p.chunks0 + p.chunks1) <= 4;
  if (store_heavy) {
    if (block_n == 256) return launch<256, 0, 1>(ma0, ma1, mb, mo, p, sms, st);
    if (block_n == 128) return launch<128, 0, 1>(ma0, ma1, mb, mo, p, sms, st);
    return launch<64, 0, 1>(ma0, ma1, mb, mo, p, sms, st);
  }
  if (use_pair && block_n == 256) {
    if (!stats) return launch_pair<256, 0>(ma0, ma1, mb, mo, p, sms, st);
    return p.n_tiles == 1 ? launch_pair<256, 8>(ma0, ma1, mb, mo, p, sms, st) : launch_pair<256, 4>(ma0, ma1, mb, mo, p, sms, st);
  }
  if (use_pair) {
    // four M-tiles per pair (two per CTA) when the M-tile count allows it
    const bool mt2 = ((long)p.N * p.tiles_w * p.tiles_h) % 4 == 0 && p.total_tiles >= 4;
    if (mt2) return stats ? launch_pair<128, 8, 2>(ma0, ma1, mb, mo, p, sms, st) : launch_pair<128, 0, 2>(ma0, ma1, mb, mo, p, sms, st);
    return stats ? launch_pair<128, 8>(ma0, ma1, mb, mo, p, sms, st) : launch_pair<128, 0>(ma0, ma1, mb, mo, p, sms, st);
  }
  if (block_n == 256) {
    if (!stats) return launch<256, 0>(ma0, ma1, mb, mo, p, sms, st);
    return p.n_tiles == 1 ? launch<256, 8>(ma0, ma1, mb, mo, p, sms, st) : launch<256, 4>(ma0, ma1, mb, mo, p, sms, st);
  }
  if (block_n == 128) return stats ? launch<128, 8>(ma0, ma1, mb, mo, p, sms, st) : launch<128, 0>(ma0, ma1, mb, mo, p, sms, st);
  return stats ? launch<64, 8>(ma0, ma1, mb, mo, p, sms, st) : launch<64, 0>(ma0, ma1, mb, mo, p, sms, st);
}
