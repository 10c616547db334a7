// Weight gradient of the UNet convolutions (the autograd backward of every nn.Conv2d /
// WeightStandardizedConv2d call of denoising_diffusion.py:92,98,114,200,222,225,253,254,297,339,354)
// on the tcgen05 tensor cores.
//
//   dW[co][tap*Cin + ci] = sum over pixels  src[n, h+dy(tap), w+dx(tap), ci] * dy[n, h, w, co]
//
//   GEMM view:  M = 128 input channels (two 64-channel chunks of the concatenated sources),
//               N = BN output channels (64 / 128 / 256),
//               K = pixels, consumed 64 at a time (one TMA box per 64-channel chunk), one job per tap.
//
//   Both operands are bf16 NHWC, so the reduction dimension (pixels) is the STRIDED one: the tiles are
//   "MN-major" UMMA operands.  The very TMA box the forward kernel uses as a K-major A tile, {64 ch, Wt, R}
//   with the 128-byte swizzle, is also the canonical MN-major SWIZZLE_128B layout -- 8 pixel rows x 128 B per
//   swizzle atom, atoms of successive 8-pixel groups 1024 B apart (SBO), successive 64-channel chunks one box
//   apart (LBO) -- so wgrad needs no transposed copy of either tensor: the instruction descriptor just sets
//   a_major = b_major = MN.  The tap shift and the zero padding are again the TMA box origin and its
//   out-of-bounds zero fill.
//
//   Job = (64-pixel tile range, tap, BN output channels, 128 input channels); one CTA per job, fp32 accumulator
//   in TMEM for the whole range, then the 128 x BN block is added into dW with coalesced fp32 atomics (lanes =
//   consecutive ci).  Jobs that share a pixel range are adjacent in blockIdx so they run together and the
//   activation tiles are served by L2.
#include "fd_tc.cuh"

using namespace fdtc;

namespace {

constexpr int kPx = 64;                       // pixels per K-block
constexpr int kChunkBytes = kPx * 128;        // one {64 ch, 64 px} box: 8 KiB
constexpr int kThreads = 192;                 // warp 0 TMA, warp 1 MMA, warps 2..5 epilogue

struct WgradParams {
  int N, H, W;               // geometry of dy (after flattening / merging)
  int Cout, Cin;
  int KW, taps, pad_h, pad_w, mode;
  int chunks0, chunks;       // 64-channel chunks of src0 / of src0+src1
  int R, Wt, tiles_w, tiles_h, total_tiles;
  int ci_blks, co_blks, splits;
  float* dw;
};

template <int BN>
struct WCfg {
  static constexpr int kABytes = 2 * kChunkBytes;
  static constexpr int kBBytes = (BN / 64) * kChunkBytes;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = BN == 256 ? 4 : (BN == 128 ? 6 : 8);
  static constexpr int kTmemCols = BN < 32 ? 32 : BN;
  static constexpr int kSmemBytes = 1024 + kStages * kStageBytes + 256;
};

// MN-major SWIZZLE_128B operand: 64-element (128 B) rows along MN, 8 K-rows per atom, K groups SBO = 1024 B apart,
// 64-element MN chunks `lbo` bytes apart.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t saddr, uint32_t lbo) {
  uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(lbo >> 4) << 16;
  d |= (uint64_t)(1024u >> 4) << 32;
  d |= 1ull << 46;
  d |= 2ull << 61;
  return d;
}
// D fp32, A/B bf16, both MN-major
__host__ __device__ constexpr uint32_t umma_idesc_bf16_mn(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

template <int BN>
__global__ void __launch_bounds__(kThreads, 1)
conv_wgrad_kernel(const __grid_constant__ CUtensorMap map_a0, const __grid_constant__ CUtensorMap map_a1,
                  const __grid_constant__ CUtensorMap map_dy, const WgradParams p) {
  using C = WCfg<BN>;
  constexpr int STAGES = C::kStages;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t bar_base = base + STAGES * C::kStageBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  const uint32_t done_bar = bar_base + 8u * (2 * STAGES);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(gbase + STAGES * C::kStageBytes + 8 * (2 * STAGES + 1) + 8);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // job decode: ci block fastest, then co block, tap, pixel split (jobs sharing a pixel range are neighbours)
  int id = blockIdx.x;
  const int ci_blk = id % p.ci_blks; id /= p.ci_blks;
  const int co_blk = id % p.co_blks; id /= p.co_blks;
  const int tap = id % p.taps;
  const int split = id / p.taps;
  const int t_begin = (int)(((long)p.total_tiles * split) / p.splits);
  const int t_end = (int)(((long)p.total_tiles * (split + 1)) / p.splits);
  const int nchunk = (p.chunks - 2 * ci_blk) >= 2 ? 2 : 1;      // 64-channel chunks this job really owns
  const int tiles_per_img = p.tiles_w * p.tiles_h;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a0);
    tma_prefetch_desc(&map_a1);
    tma_prefetch_desc(&map_dy);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(done_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(s_tmem), C::kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;

  if (warp == 0) {
    if (elect_one_sync()) {
      int stage = 0;
      uint32_t phase = 0;
      const int ky = tap / p.KW, kx = tap - ky * p.KW;
      for (int t = t_begin; t < t_end; ++t) {
        const int img = t / tiles_per_img;
        const int rem = t - img * tiles_per_img;
        const int h0 = (rem / p.tiles_w) * p.R;
        const int w0 = (rem % p.tiles_w) * p.Wt;
        mbar_wait(empty_bar(stage), phase ^ 1u);
        mbar_expect_tx(full_bar(stage), (uint32_t)(nchunk + BN / 64) * kChunkBytes);
        const uint32_t dst_a = base + stage * C::kStageBytes;
        const uint32_t dst_b = dst_a + C::kABytes;
        for (int a = 0; a < nchunk; ++a) {
          const int chunk = 2 * ci_blk + a;
          const CUtensorMap* ma = chunk < p.chunks0 ? &map_a0 : &map_a1;
          const int c0 = (chunk < p.chunks0 ? chunk : chunk - p.chunks0) * 64;
          if (p.mode == 0)
            tma_load_5d(dst_a + a * kChunkBytes, ma, full_bar(stage), c0, w0 + kx - p.pad_w, h0 + ky - p.pad_h, img, 0);
          else
            tma_load_5d(dst_a + a * kChunkBytes, ma, full_bar(stage), c0, tap & 1, w0, tap >> 1, h0);
        }
#pragma unroll
        for (int b = 0; b < BN / 64; ++b)
          tma_load_5d(dst_b + b * kChunkBytes, &map_dy, full_bar(stage), co_blk * BN + b * 64, w0, h0, img, 0);
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // one elected lane runs the whole loop; the next stage's barrier wait and descriptor bases (general registers) come before
    // this stage's commit so that only register-to-uniform moves separate two stages' MMAs (see conv_igemm_kernel)
    constexpr uint32_t idesc = umma_idesc_bf16_mn(128, BN);
    if (elect_one_sync()) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t lbo_a = nchunk == 2 ? (uint32_t)kChunkBytes : 0u;   // single chunk: rows 64..127 alias rows 0..63 (ignored)
      const uint64_t adesc0 = umma_desc_mn_sw128(base, lbo_a);
      const uint64_t bdesc0 = umma_desc_mn_sw128(base + C::kABytes, (uint32_t)kChunkBytes);
      uint64_t ad = opaque64(adesc0), bd = opaque64(bdesc0);
      bool waited = false;
      for (int t = t_begin; t < t_end; ++t) {
        if (!waited) mbar_wait(full_bar(stage), phase);
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < kPx / 16; ++k) {
          // 16 pixels = two 8-row swizzle atoms = 2048 B further along K (+128 in the address field)
          umma_bf16(tmem_base, ad + (uint64_t)(k * (2048 >> 4)), bd + (uint64_t)(k * (2048 >> 4)), idesc,
                    (t != t_begin || k != 0) ? 1u : 0u);
        }
        const uint32_t cur_empty = empty_bar(stage);
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        ad = opaque64(adesc0 + (uint64_t)(stage * (C::kStageBytes >> 4)));
        bd = opaque64(bdesc0 + (uint64_t)(stage * (C::kStageBytes >> 4)));
        waited = t + 1 < t_end;
        if (waited) mbar_wait(full_bar(stage), phase);
        umma_commit(cur_empty);
        if (t == t_end - 1) umma_commit(done_bar);
      }
    }
    __syncwarp();
  } else if (t_end > t_begin) {
    // epilogue: TMEM lane = input channel row, column = output channel
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int a = row >> 6;
    mbar_wait(done_bar, 0);
    tc_fence_after();
    if (a < nchunk) {
      const int ci = (2 * ci_blk + a) * 64 + (row & 63);
      const long ktot = (long)p.taps * p.Cin;
      float* dst = p.dw + (long)(co_blk * BN) * ktot + (long)tap * p.Cin + ci;
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        uint32_t acc[32];
        tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(c * 32), acc);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) atomicAdd(dst + (long)(c * 32 + j) * ktot, __uint_as_float(acc[j]));
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::kTmemCols);
  }
}

struct Tile64 {
  int R, Wt;
};

Tile64 pick_tile64(int H, int W) {
  Tile64 best{1, 64};
  long best_cost = -1;
  for (int wt = 64; wt >= 8; wt >>= 1) {
    const int r = kPx / wt;
    const long cost = (long)((W + wt - 1) / wt) * wt * (long)((H + r - 1) / r) * r;
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best = Tile64{r, wt};
    }
  }
  return best;
}

template <int BN>
int launch_wgrad(const CUtensorMap& ma0, const CUtensorMap& ma1, const CUtensorMap& mdy, const WgradParams& p, int grid,
                 cudaStream_t st) {
  using C = WCfg<BN>;
  static bool attr_set = false;
  if (!attr_set) {
    FD_CUDA(cudaFuncSetAttribute(conv_wgrad_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmemBytes));
    attr_set = true;
  }
  conv_wgrad_kernel<BN><<<grid, kThreads, C::kSmemBytes, st>>>(ma0, ma1, mdy, p);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

}  // namespace

// fd_conv_wgrad_strip.cu
int fd_conv_wgrad_strip_launch(const void* src0, int C0, const void* src1, int C1, const void* dy, float* dw, int N, int H,
                               int W, int Cout, void* stream);

extern "C" {

int fd_conv_wgrad(const void* src0, int C0, const void* src1, int C1, const void* dy, float* dw, int N, int H, int W,
                  int Cout, int KH, int KW, int pad_h, int pad_w, int mode, void* stream) {
  FD_REQUIRE(src0 && dy && dw, "conv_wgrad: null pointer");
  FD_REQUIRE(N > 0 && H > 0 && W > 0, "conv_wgrad: bad geometry N=%d H=%d W=%d", N, H, W);
  FD_REQUIRE(C0 > 0 && C0 % 64 == 0 && C1 >= 0 && C1 % 64 == 0, "conv_wgrad: C0=%d C1=%d must be multiples of 64", C0, C1);
  FD_REQUIRE(src1 != nullptr || C1 == 0, "conv_wgrad: C1 > 0 needs src1");
  FD_REQUIRE(Cout > 0 && Cout % 64 == 0, "conv_wgrad: Cout=%d must be a multiple of 64", Cout);
  FD_REQUIRE(mode == 0 || mode == 1, "conv_wgrad: mode %d", mode);
  FD_REQUIRE(mode == 0 || C1 == 0, "conv_wgrad: mode 1 takes one source");
  FD_REQUIRE(KH >= 1 && KW >= 1 && KH * KW <= 64, "conv_wgrad: bad kernel %dx%d", KH, KW);
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    FD_CUDA(cudaGetDevice(&dev));
    FD_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  }
  if (mode == 0 && KH == 3 && KW == 3 && pad_h == 1 && pad_w == 1 && W >= 64 && Cout <= 128) {
    // rolling-strip kernel: every source / dy row is loaded once instead of once per tap (measured: 800-880 TFLOP/s vs
    // 140-410 for Cout <= 128; the N = 256 tiles of the generic kernel stay ahead for Cout >= 256: 700-800 vs 630-650)
    return fd_conv_wgrad_strip_launch(src0, C0, src1, C1, dy, dw, N, H, W, Cout, stream);
  }
  WgradParams p{};
  p.Cout = Cout;
  p.Cin = C0 + C1;
  p.mode = mode;
  p.chunks0 = C0 / 64;
  p.chunks = (C0 + C1) / 64;
  p.dw = dw;
  CUtensorMap ma0, ma1, mdy;
  Tile64 ts;
  if (mode == 0) {
    int n = N, h = H, w = W;
    if (KH == 1 && KW == 1 && pad_h == 0 && pad_w == 0) {   // 1x1: the whole batch is one row of pixels
      FD_REQUIRE((long)N * H * W < (1L << 31), "conv_wgrad: too many pixels");
      w = N * H * W;
      h = 1;
      n = 1;
    }
    p.N = n; p.H = h; p.W = w;
    p.KW = KW;
    p.taps = KH * KW;
    p.pad_h = pad_h;
    p.pad_w = pad_w;
    ts = pick_tile64(h, w);
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
    p.N = 1; p.H = N * H; p.W = W;
    p.KW = 2;
    p.taps = 4;
    ts = pick_tile64(p.H, p.W);
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
  const long total = (long)p.N * p.tiles_w * p.tiles_h;
  FD_REQUIRE(total < (1L << 31), "conv_wgrad: too many tiles");
  p.total_tiles = (int)total;
  {
    const uint64_t dims[5] = {(uint64_t)Cout, (uint64_t)p.W, (uint64_t)p.H, (uint64_t)p.N, 1};
    const uint64_t str[4] = {(uint64_t)Cout * 2, (uint64_t)p.W * Cout * 2, (uint64_t)p.H * p.W * Cout * 2,
                             (uint64_t)p.N * p.H * p.W * Cout * 2};
    const uint32_t box[5] = {64, (uint32_t)ts.Wt, (uint32_t)ts.R, 1, 1};
    if (int e = make_tmap_bf16(&mdy, dy, 5, dims, str, box)) return e;
  }
  const int bn = (Cout % 256 == 0) ? 256 : ((Cout % 128 == 0) ? 128 : 64);
  p.ci_blks = (p.chunks + 1) / 2;
  p.co_blks = Cout / bn;
  const long base_jobs = (long)p.ci_blks * p.co_blks * p.taps;
  // pixel splits: about two waves of CTAs, at least 4 K-blocks per job
  long splits = (2L * sms + base_jobs - 1) / base_jobs;
  if (splits > total / 4) splits = total / 4;
  if (splits < 1) splits = 1;
  p.splits = (int)splits;
  const long grid = base_jobs * splits;
  FD_REQUIRE(grid < (1L << 31), "conv_wgrad: too many jobs");
  cudaStream_t st = (cudaStream_t)stream;
  if (bn == 256) return launch_wgrad<256>(ma0, ma1, mdy, p, (int)grid, st);
  if (bn == 128) return launch_wgrad<128>(ma0, ma1, mdy, p, (int)grid, st);
  return launch_wgrad<64>(ma0, ma1, mdy, p, (int)grid, st);
}

}  // extern "C"
