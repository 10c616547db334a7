// 3x3 / pad 1 / 64 -> 64 channel convolution for large images (the full-resolution ResnetBlock convs of the
// UNet, denoising_diffusion.py:172-214: 8 launches and 15 % of the forward FLOPs at 440x1024).
//
// The generic implicit GEMM (fd_conv_igemm.cu) re-reads every input pixel once per tap and the weights once
// per tile: 216 KB of L2->smem traffic per 9.4 MFLOP tile, which bounds it at ~0.45 PFLOP/s.  Here
//   * the 72 KB of packed weights are loaded ONCE per CTA and stay resident in shared memory;
//   * a CTA walks down a column strip of the image (128 output pixels wide, SEG rows tall).  Input rows are
//     TMA-loaded once as 130-pixel strips (left/right halo included; rows / columns outside the image are
//     zero-filled by TMA) into a 5-slot ring; the 9 taps of an output row are 9 UMMA A-operands that alias
//     three strips at a 0/1/2-pixel (0/128/256-byte) offset -- no data is re-fetched or re-arranged;
//   * so each output row costs one new 16.6 KB strip: ~13x less L2 traffic, the kernel becomes MMA/epilogue bound.
// Warp roles and the epilogue (GroupNorm partial sums, swizzled smem + TMA store) are those of the generic kernel.
//
// 128 input channels (the skip-concat convs ups.3.x / final_res_block, and the upsample conv ups.2.3) run as TWO
// passes of this kernel, one per 64-channel half: pass 1 writes the partial sum to `out`, pass 2 adds it back as
// its residual (same tile reads then overwrites the same rows) and produces bias + statistics.  Streaming the
// 144 KB of weights per tile instead was measured to be no faster than the generic kernel (chip-level L2->SM
// bandwidth), while two resident-weight passes cost 0.75 ms instead of 1.09 ms.
//
// The MMA issuer stages the strips in tensor memory (tcgen05.cp) and issues the A-from-TMEM ("TS") form of tcgen05.mma.  An
// earlier issuer fed both MMA operands from shared memory ("SS"); it was shared-memory-bandwidth bound as analysed below, and
// the TS form removes three quarters of those operand reads (see the issuer branch).
//
// Where the time went in the SS variant (ncu + scripts/micro/umma_rate.cu, profiles/r1_umma_rate.txt): an SS-mode 128xNx16 UMMA reads
// (128 + N) * 32 bytes of shared memory at 128 B/clk, so an N = 64 instruction takes 48 cycles, not 32.  Per 128-pixel tile
// the 36 MMAs read 216 KB, TMA writes 16.6 KB, the epilogue writes and the TMA store reads 16 KB each: 265 KB = 2070
// cycles of the shared-memory pipe out of the 2680 the tile takes (l1tex throughput 77 %, tensor pipe "active" 51 %).
// The kernel is shared-memory-bandwidth bound.  Tried and measured slower (0.387 vs 0.268 ms for 64->64 at 8x440x1024):
// one N = 192 instruction per kernel row on the unshifted strip with the kx shift done in the epilogue by warp shuffles --
// 44 % less operand traffic, but 192 accumulator columns leave room for only two TMEM stages and the longer epilogue
// (3 x tcgen05.ld, quarter-to-quarter row exchange) then sits on the critical path.
#include "fd_conv_epi.cuh"

using namespace fdtc;

namespace {

constexpr int kC = 64;                         // input = output channels
constexpr int kTileW = 128;                    // output pixels per tile (one image row segment)
constexpr int kStripPx = kTileW + 2;           // + left/right halo
constexpr int kStripTx = kStripPx * 128;       // bytes TMA delivers per strip
constexpr int kStripBytes = 136 * 128;         // slot size: multiple of 1024 keeps the swizzle phase of every slot
constexpr int kNS = 5;                         // strips in flight: 3 in use + 2 prefetched (6 measured no faster)
constexpr int kWTapBytes = kC * kC * 2;        // one tap of weights: [64 cout][64 cin] bf16
constexpr int kWBytes = 9 * kWTapBytes;        // 72 KB, resident
constexpr int kThreads = 64 + kEpiThreads + 64;  // warp 0 TMA, warp 1 MMA issuer, warps 2..9 epilogue; warps 10, 11: the input
                                                 // transform of the fused GroupNorm + SiLU variant
constexpr int kTail = 256 + 2 * kC * 4 + kEpiWarps * 16 * 4 + 64;
constexpr int kSmemBytes = 1024 + kWBytes + kNS * kStripBytes + 2 * kSlabBytes + kTail;

// A operand from tensor memory ("TS" form): staged there by tcgen05.cp, which reads the same canonical K-major SWIZZLE_128B
// shared-memory layout as the SS-form instruction (scripts/micro/umma_ts.cu: bit-identical products, also with the start
// shifted by whole 128-byte pixel rows; 32.0 cycles per 128x64x16 instruction instead of 48.0)
__device__ __forceinline__ void utccp_128x256b(uint32_t tmem_dst, uint64_t sdesc) {
  asm volatile("tcgen05.cp.cta_group::1.128x256b [%0], %1;" ::"r"(tmem_dst), "l"(sdesc) : "memory");
}
__device__ __forceinline__ void umma_ts_bf16(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
constexpr int kATmemCol0 = 2 * kC;             // accumulators in columns [0, 128), A ring in [128, 512)
constexpr int kATmemSlotCols = 3 * (kC / 2);   // one strip = 3 kx-shifted copies x 32 columns (64 bf16 per lane)
constexpr int kATmemSlots = 4;                 // 3 strips in use + 1 being staged

// silu(z) = z sigmoid(z) = h + h tanh(h), h = z / 2: ONE MUFU op (tanh.approx, 2^-11 relative) instead of the ex2 + rcp of
// (Round 2: FOUR transform warps, one per scheduler / MUFU unit, with their own 14-warp template variant, made the fused launch
// faster when timed alone -- conv roofline fraction 0.80-0.83 vs 0.77-0.79 -- and left DDIM-50 unchanged on the same box,
// 9.53 vs 9.51 flows/s (two builds alternated on one box): the board is power-capped, the step is energy-bound.  Not kept.)
// fd_silu.  The fused input transform runs on two warps = two of the SM's four MUFU units; with two MUFU ops per element it
// needed ~2100 cycles per strip (more than a tile's MMAs), with one ~1050.  The result differs from fd_silu by < 2^-10
// relative before the bf16 rounding (2^-9) that follows.
__device__ __forceinline__ float silu_tanh(float z) {
  const float h = 0.5f * z;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}

struct StripParams {
  int N, H, W;
  int wblocks, total_rows;   // column blocks per image; N * wblocks * H output rows in (image, column block, row) order
  int tile_w;                // output pixels per tile
  int c_off;                 // first input channel of this pass inside the source tensor (0 or 64)
  int w_k0, w_kstride;       // weight K coordinate of tap t = t * w_kstride + w_k0
  const float* bias;
  const __nv_bfloat16* residual;
  double* gn_stats;
  // fused input transform: the strips are activated in shared memory, x -> silu(a[c] x + b[c]) with the
  // GroupNorm statistics of the INPUT tensor folded into a, b exactly as gn_silu_kernel does (Block.forward :176-187)
  const double* in_stats;    // [N][8][2] or null (no transform)
  const float* in_gamma;
  const float* in_beta;
  const float* in_ss;        // (scale | shift) rows or null
  long in_ss_stride;
  float in_eps;
  int dbg;                   // FD_CONV_DBG in FD_DIAG builds: 4 = no MMAs, 8 = epilogue handshakes only, 64 = no tcgen05.cp
};

// Work split: the N * wblocks * H output rows (128-pixel tiles), ordered (image, column block, row), are cut into gridDim.x
// equal contiguous ranges, one per CTA.  A CTA walks its range as 1-3 runs of consecutive rows of one column ("items");
// every run costs two extra halo strips, so long runs are cheap, and the ranges differ by at most one tile (the former
// round-robin over 16..64-row segments left 180 vs 200 tiles on different SMs and paid the halo ten times per CTA).
struct StripWalk {
  int cur, end;
  __device__ __forceinline__ explicit StripWalk(const StripParams& p) {
    cur = (int)((long)p.total_rows * blockIdx.x / gridDim.x);
    end = (int)((long)p.total_rows * (blockIdx.x + 1) / gridDim.x);
  }
  __device__ __forceinline__ bool next(const StripParams& p, int& n, int& w0, int& ra, int& rb) {
    if (cur >= end) return false;
    const int col = cur / p.H;
    ra = cur - col * p.H;
    const int rows = min(p.H - ra, end - cur);
    rb = ra + rows;
    n = col / p.wblocks;
    w0 = (col - n * p.wblocks) * p.tile_w;
    cur += rows;
    return true;
  }
};

// Epilogue of the classic (nine N = 64 taps) variant.  Measured: with all 8 epilogue warps working on ONE tile the
// kernel spends ~2800 cycles per tile although the MMAs need 1728 and the epilogue only issues ~700 cycles' worth of
// instructions (ncu: issue active 22 %) -- it is bound by the LATENCY of the dependent chain tcgen05.ld -> math ->
// st.shared -> fence -> barrier -> TMA store.  So the 8 warps form TWO groups of 4 (one warp per TMEM lane quarter,
// 64 columns per thread) that drain alternating tiles = alternating TMEM stages, each with its own staging slab and
// named barrier: two tiles are in flight in the epilogue, like the two MMA issuer warps upstream.
template <int GPT, class NextTile>
__device__ __forceinline__ void strip_epilogue2(const EpiCtx& ec, NextTile next_tile) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ew = warp - 2;
  const int quarter = warp & 3, group = ew >> 2;
  const int gt = (ew & 3) * 32 + lane;               // thread index inside the group: 0..127
  const int row = quarter * 32 + lane;
  const int bar_id = 1 + group;
  float* const bias_s = ec.s_bias + group * kC;
  float* const s_stats = ec.s_stats + group * 64;    // [4 warps][16]
  constexpr int NG = GPT > 0 ? GPT : 1;
  constexpr int CPG = kC / 8;                        // 8 channels per group
  float st_s[NG], st_q[NG];
#pragma unroll
  for (int b = 0; b < NG; ++b) st_s[b] = st_q[b] = 0.f;
  int st_img = -1;
  const uint32_t buf = ec.o_smem + group * kSlabBytes;
  if (gt < kC) bias_s[gt] = ec.bias ? __ldg(ec.bias + gt) : 0.f;
  named_bar_sync(bar_id, 128);

  auto flush_stats = [&]() {
    if (GPT == 0 || st_img < 0) return;
    float* mine = s_stats + (ew & 3) * 16;
#pragma unroll
    for (int b = 0; b < NG; ++b) {
      const float s = fd_warp_sum(st_s[b]), q = fd_warp_sum(st_q[b]);
      if (lane == 0) {
        mine[b * 2] = s;
        mine[b * 2 + 1] = q;
      }
      st_s[b] = st_q[b] = 0.f;
    }
    named_bar_sync(bar_id, 128);
    if (gt < 2 * GPT) {
      const float sv = (s_stats[gt] + s_stats[16 + gt]) + (s_stats[32 + gt] + s_stats[48 + gt]);     // fixed order
      atomicAdd(ec.gn_stats + (long)st_img * 16 + gt, (double)sv);
    }
    named_bar_sync(bar_id, 128);
  };

  EpiTile tc;
  for (int iter = 0; next_tile(iter, tc); ++iter) {
    if ((iter & 1) != group) continue;
    const int as = group;
    const uint32_t aphase = (iter >> 1) & 1;
    const int img = tc.img, h = tc.h0, w0 = tc.w0;
    const int w = w0 + row;
    const bool valid = w < ec.W;
    if (GPT > 0 && img != st_img) {
      flush_stats();
      st_img = img;
    }
    mbar_wait(ec.tfull0 + 8u * as, aphase);
    tc_fence_after();
    if (kDiag && (ec.dbg & 8)) {
      tc_fence_before();
      mbar_arrive(ec.tempty0 + 8u * as);
      continue;
    }
    uint32_t acc[2][32];
    const uint32_t taddr = ec.tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(as * kC);
    tmem_ld32(taddr, acc[0]);
    tmem_ld32(taddr + 32, acc[1]);
    tmem_ld_wait();
    tc_fence_before();
    mbar_arrive(ec.tempty0 + 8u * as);
    const long pix = ((long)img * ec.H + h) * ec.W + w;
    uint32_t packed[32];
#pragma unroll
    for (int hc = 0; hc < 2; ++hc) {
      float v[32];
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4) {
        const float4 b4 = *reinterpret_cast<const float4*>(bias_s + hc * 32 + j4 * 4);
        v[j4 * 4 + 0] = __uint_as_float(acc[hc][j4 * 4 + 0]) + b4.x;
        v[j4 * 4 + 1] = __uint_as_float(acc[hc][j4 * 4 + 1]) + b4.y;
        v[j4 * 4 + 2] = __uint_as_float(acc[hc][j4 * 4 + 2]) + b4.z;
        v[j4 * 4 + 3] = __uint_as_float(acc[hc][j4 * 4 + 3]) + b4.w;
      }
      if (ec.residual != nullptr && valid) {
        const __nv_bfloat16* rrow = ec.residual + pix * kC + hc * 32;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint4 r4 = __ldg(reinterpret_cast<const uint4*>(rrow) + q);
          const uint32_t rw[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 f = fd_unpack_bf16(rw[e]);
            v[q * 8 + e * 2] += f.x;
            v[q * 8 + e * 2 + 1] += f.y;
          }
        }
      }
      if (GPT > 0 && valid) {
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          float s = 0.f, q = 0.f;
#pragma unroll
          for (int j = 0; j < CPG; ++j) {
            const float x = v[b * CPG + j];
            s += x;
            q = fmaf(x, x, q);
          }
          st_s[(hc * 4 + b) % NG] += s;
          st_q[(hc * 4 + b) % NG] += q;
        }
      }
#pragma unroll
      for (int j = 0; j < 16; ++j) packed[hc * 16 + j] = fd_pack_bf16(v[2 * j], v[2 * j + 1]);
    }
    if ((ew & 3) == 0 && elect_one_sync()) tma_store_wait_read<0>();   // this group's previous store has read the slab
    named_bar_sync(bar_id, 128);
    const uint32_t rbase = buf + (uint32_t)row * 128u;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const uint32_t piece = (uint32_t)q ^ (uint32_t)(row & 7);
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(rbase + piece * 16u), "r"(packed[q * 4]),
                   "r"(packed[q * 4 + 1]), "r"(packed[q * 4 + 2]), "r"(packed[q * 4 + 3])
                   : "memory");
    }
    fence_proxy_async_smem();
    named_bar_sync(bar_id, 128);
    if ((ew & 3) == 0 && elect_one_sync()) {             // the group's first warp; elect.sync keeps UTMASTG straight-line
      tma_store_5d(ec.map_out, buf, 0, w0, h, img, 0);
      tma_store_commit();
    }
  }
  flush_stats();
  __syncwarp();
  if ((ew & 3) == 0 && elect_one_sync()) tma_store_wait_all();
}

template <int GPT>
__global__ void __launch_bounds__(kThreads, 1)
conv3x3_strip_kernel(const __grid_constant__ CUtensorMap map_in, const __grid_constant__ CUtensorMap map_w,
                     const __grid_constant__ CUtensorMap map_out, const StripParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t w_smem = base;
  const uint32_t s_smem = base + kWBytes;
  const uint32_t o_smem = s_smem + kNS * kStripBytes;
  const uint32_t bar_base = o_smem + 2 * kSlabBytes;
  const uint32_t wfull_bar = bar_base;
  auto full_bar = [&](int s) { return bar_base + 8u * (1 + s); };
  auto empty_bar = [&](int s) { return bar_base + 8u * (1 + kNS + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (1 + 2 * kNS + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (3 + 2 * kNS + s); };
  auto xfull_bar = [&](int s) { return bar_base + 8u * (5 + 2 * kNS + s); };   // strip transformed (fused GroupNorm input)
  const bool fuse_in = p.in_stats != nullptr;
  uint8_t* gtail = gbase + kWBytes + kNS * kStripBytes + 2 * kSlabBytes + 256;
  float* s_bias = reinterpret_cast<float*>(gtail);
  float* s_stats = reinterpret_cast<float*>(gtail + 2 * kC * 4);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(gtail + 2 * kC * 4 + kEpiWarps * 16 * 4);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_in);
    tma_prefetch_desc(&map_w);
    tma_prefetch_desc(&map_out);
    mbar_init(wfull_bar, 1);
    for (int s = 0; s < kNS; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
      mbar_init(xfull_bar(s), 64);        // the two transform warps
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), 128);      // each accumulator stage is drained by one group of 4 epilogue warps
    }
    fence_barrier_init();
  }
  constexpr uint32_t kTmemCols = 512;
  if (warp == 1) tmem_alloc(smem_u32(s_tmem), kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;

  if (warp == 0) {
    // ===================== TMA producer: weights once, then one strip per input row =====================
    if (elect_one_sync()) {
      mbar_expect_tx(wfull_bar, kWBytes);
      for (int tap = 0; tap < 9; ++tap)
        tma_load_2d(w_smem + tap * kWTapBytes, &map_w, wfull_bar, tap * p.w_kstride + p.w_k0, 0);
      uint32_t seq = 0;
      StripWalk walk(p);
      int n, w0, ra, rb;
      while (walk.next(p, n, w0, ra, rb)) {
        for (int y = ra - 1; y <= rb; ++y, ++seq) {
          const int slot = seq % kNS;
          const uint32_t phase = (seq / kNS) & 1u;
          mbar_wait(empty_bar(slot), phase ^ 1u);
          mbar_expect_tx(full_bar(slot), kStripTx);
          tma_load_5d(s_smem + slot * kStripBytes, &map_in, full_bar(slot), p.c_off, w0 - 1, y, n, 0);
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer, A operand from tensor memory =====================
    // The SS form reads (128 + 64) * 32 B of shared memory per 128x64x16 instruction = 48 cycles at 128 B/clk, and the nine
    // taps re-read every strip nine times: 216 KB per tile, which made this kernel shared-memory bound (file header).  Here
    // every input strip is copied to tensor memory ONCE per kx shift (tcgen05.cp.128x256b, 12 copies = 48 KB of reads per
    // strip), a 4-slot ring of 96 columns, and the 36 MMAs of a tile read only their 2 KB weight slices from shared memory:
    // 72 + 48 KB per tile instead of 216, and the instruction runs at the tensor rate (32 cycles).  tcgen05.cp and
    // tcgen05.mma issued by one thread execute in issue order, so the ring needs no barriers of its own; a strip's
    // shared-memory slot is handed back to the TMA producer by a commit right after its copies.
    if (elect_one_sync()) {
      constexpr uint32_t idesc = umma_idesc_bf16(kBlockM, kC);
      mbar_wait(wfull_bar, 0);
      tc_fence_after();
      const uint64_t bdesc0 = umma_desc_sw128(w_smem);
      const uint32_t a_tmem0 = tmem_base + kATmemCol0;
      // copy cursor: walks the same (item, row) sequence as the TMA producer, `cseq` = strips staged so far
      StripWalk cwalk(p);
      int c_left = 0;
      uint32_t cseq = 0;
      // "the strip is ready": landed (TMA) or, with the fused input transform, landed and activated
      auto ready_bar = [&](uint32_t slot) { return fuse_in ? xfull_bar(slot) : full_bar(slot); };
      auto copy_strip = [&]() {
        const uint32_t slot = cseq % kNS;
        mbar_wait(ready_bar(slot), (cseq / kNS) & 1u);
        tc_fence_after();
        const uint32_t dst = a_tmem0 + (cseq % kATmemSlots) * kATmemSlotCols;
        const uint64_t sd = umma_desc_sw128(s_smem + slot * kStripBytes);
#pragma unroll
        for (int kx = 0; kx < 3; ++kx)
#pragma unroll
          for (int k = 0; k < kC / 16; ++k)
            if (!(kDiag && (p.dbg & 64)))
            utccp_128x256b(dst + kx * (kC / 2) + k * 8, sd + (uint64_t)(kx * 8 + 2 * k));   // +8: one 128-byte pixel row
        umma_commit(empty_bar(slot));
        ++cseq;
      };
      auto strips_left = [&]() {                     // is there another strip in this CTA's sequence?
        while (c_left == 0) {
          int cn, cw0, cra, crb;
          if (!cwalk.next(p, cn, cw0, cra, crb)) return false;
          c_left = crb - cra + 2;
        }
        return true;
      };
      // The thread that issues the MMAs is held back by the tensor pipe while a tile's 36 instructions drain, and everything it
      // does BETWEEN two tiles is time the pipe sits empty (probes in a diagnostic build: 1333 cycles of issue per tile = the
      // hardware rate, plus ~250 cycles deciding about the next strip, ~90 waiting for the accumulator stage, ~290 of loop
      // bookkeeping).  So the next tile is prepared in the middle of the current tile's instruction stream (after MMA 24):
      // advance the cursor, wait for the next accumulator stage, claim the next strip and test whether it has landed.
      struct Claim {
        bool more, inter;          // a strip is staged during this tile / its data had landed when the tile started
        uint32_t slot, phase, dst;
        uint64_t sd;
      };
      auto claim = [&](uint32_t f) {          // f = first strip of the tile during which the claimed strip is staged
        Claim c{};
        c.more = cseq < f + 4 && strips_left();
        if (c.more) {
          c.slot = cseq % kNS;
          c.phase = (cseq / kNS) & 1u;
          c.dst = a_tmem0 + (cseq % kATmemSlots) * kATmemSlotCols;
          c.sd = umma_desc_sw128(s_smem + c.slot * kStripBytes);
          ++cseq;
          --c_left;
        }
        return c;
      };
      auto landed = [&](Claim& c) { c.inter = c.more && mbar_try_wait(ready_bar(c.slot), c.phase); };
      long long dg_t0 = 0, dg_mma = 0, dg_tail = 0;
      unsigned long long dg_ns0 = 0;
      if (kDiag) {
        dg_t0 = clock64();
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dg_ns0));
      }
      StripWalk walk(p);
      int wn, ww0, wra, wrb;
      int iter = 0;
      if (walk.next(p, wn, ww0, wra, wrb)) {
        int rows = wrb - wra, j = 0;
        uint32_t f = 0;
        while (cseq < f + 3) {                      // the first three strips of the CTA
          strips_left();
          copy_strip();
          --c_left;
        }
        mbar_wait(tempty_bar(0), 1u);
        Claim cp = claim(f);
        landed(cp);
        tc_fence_after();
        while (true) {
          const int as = iter & 1;
          const uint32_t tmem_d = tmem_base + as * kC;
          bool has_next = false, boundary = false;
          uint32_t f_next = 0;
          Claim cp_next{};
          long long dg_m = 0;
          if (kDiag) dg_m = clock64();
#pragma unroll
          for (int ky = 0; ky < 3; ++ky) {
            const uint32_t a_strip = a_tmem0 + ((f + ky) % kATmemSlots) * kATmemSlotCols;
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
              const uint64_t bdesc = bdesc0 + (uint64_t)((ky * 3 + kx) * (kWTapBytes >> 4));
#pragma unroll
              for (int k = 0; k < kC / 16; ++k) {
                if (!(kDiag && (p.dbg & 4)))
                  umma_ts_bf16(tmem_d, a_strip + kx * (kC / 2) + k * 8, bdesc + (uint64_t)(2 * k), idesc, (ky | kx | k) != 0 ? 1u : 0u);
                const int m = (ky * 3 + kx) * 4 + k;
                // one staging copy after every third MMA (1332 cycles per tile against 1803 with the copies back to back)
                if (m % 3 == 2 && cp.inter && !(kDiag && (p.dbg & 64))) {
                  const int c = m / 3, ckx = c >> 2, ck = c & 3;
                  utccp_128x256b(cp.dst + ckx * (kC / 2) + ck * 8, cp.sd + (uint64_t)(ckx * 8 + 2 * ck));
                }
                // ---- the next tile is prepared in small pieces spread over this tile's instruction stream: the issuing thread
                // runs only two or three MMAs ahead of the tensor pipe (the uniform-register operands of an MMA are released at
                // dispatch), so each piece has to fit into ~60 cycles and the pieces have to be a few MMAs apart
                if (m == 5) {
                  if (j + 1 < rows) {
                    has_next = true;
                    f_next = f + 1;
                  } else if (walk.next(p, wn, ww0, wra, wrb)) {
                    has_next = boundary = true;             // next run of rows: three fresh strips, staged after this tile
                    f_next = f + 3;
                  }
                }
                if (m == 14 && has_next && !boundary) cp_next = claim(f_next);
                if (m == 23 && has_next && !boundary) mbar_wait(tempty_bar((iter + 1) & 1), (((iter + 1) >> 1) & 1) ^ 1u);
                if (m == 32 && has_next && !boundary) landed(cp_next);
              }
            }
          }
          umma_commit(tfull_bar(as));
          if (kDiag) { dg_mma += clock64() - dg_m; dg_m = clock64(); }
          if (cp.inter) {
            umma_commit(empty_bar(cp.slot));
          } else if (cp.more) {                           // the strip had not landed when the tile started
            mbar_wait(ready_bar(cp.slot), cp.phase);
            tc_fence_after();
#pragma unroll
            for (int c = 0; c < 12; ++c)
              if (!(kDiag && (p.dbg & 64))) utccp_128x256b(cp.dst + (c >> 2) * (kC / 2) + (c & 3) * 8, cp.sd + (uint64_t)((c >> 2) * 8 + 2 * (c & 3)));
            umma_commit(empty_bar(cp.slot));
          }
          if (!has_next) break;
          if (boundary) {
            rows = wrb - wra;
            j = 0;
            while (cseq < f_next + 3) {
              strips_left();
              copy_strip();
              --c_left;
            }
            mbar_wait(tempty_bar((iter + 1) & 1), (((iter + 1) >> 1) & 1) ^ 1u);
            cp_next = claim(f_next);
            landed(cp_next);
          } else {
            ++j;
          }
          tc_fence_after();
          f = f_next;
          cp = cp_next;
          ++iter;
          if (kDiag) dg_tail += clock64() - dg_m;
        }
        ++iter;
      }
      if (kDiag && (p.dbg & 128) && (blockIdx.x == 0 || blockIdx.x == 77)) {
        unsigned long long ns1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns1));
        const long long cyc = clock64() - dg_t0;
        printf("strip TS issuer block %d: %d tiles, %lld cycles (%.0f / tile): MMA stream %lld, between tiles %lld, %llu ns -> %.2f GHz\n",
               blockIdx.x, iter, cyc, (double)cyc / iter, dg_mma, dg_tail, ns1 - dg_ns0, (double)cyc / (double)(ns1 - dg_ns0));
      }
    }
    __syncwarp();
  } else if (warp == 10 || warp == 11) {
    // ===================== fused input transform: GroupNorm affine + SiLU on the landed strip, in place =====================
    // Replaces the separate gn_silu pass over the producer's output (one read + one write of the tensor) for the convs whose
    // input is only consumed here (ResnetBlock block1 -> block2, :202-214).  64 threads: thread = (8-channel granule q, row
    // r0 + 8 i); rows / pixels outside the image were zero-filled by TMA and must stay zero (the padding applies to the
    // ACTIVATED tensor), so they are skipped.  Same folded coefficients as gn_silu_kernel; the SiLU uses one MUFU op (silu_tanh).
    if (fuse_in) {
      const int tl = (warp - 10) * 32 + lane;
      const int q = tl & 7, r0 = tl >> 3;
      float a[8], b[8];
      int cur_n = -1;
      uint32_t seq = 0;
      StripWalk walk(p);
      int n, w0, ra, rb;
      while (walk.next(p, n, w0, ra, rb)) {
        if (n != cur_n) {
          cur_n = n;
          const int C = kC, cpg = C >> 3;
          const double cnt = (double)p.H * (double)p.W * cpg;
          const int g = (q * 8) / cpg;
          const double sm = p.in_stats[((long)n * 8 + g) * 2], ss = p.in_stats[((long)n * 8 + g) * 2 + 1];
          const double mean = sm / cnt;
          double var = ss / cnt - mean * mean;
          if (var < 0.0) var = 0.0;
          const float rstd = (float)(1.0 / sqrt(var + (double)p.in_eps));
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int c = q * 8 + j;
            float ga = __ldg(p.in_gamma + c) * rstd;
            float be = __ldg(p.in_beta + c) - (float)mean * ga;
            if (p.in_ss != nullptr) {
              const float sc = __ldg(p.in_ss + (long)n * p.in_ss_stride + c) + 1.f;
              const float sh = __ldg(p.in_ss + (long)n * p.in_ss_stride + C + c);
              ga *= sc;
              be = be * sc + sh;
            }
            a[j] = 0.5f * ga;             // halved: the transform works on h = z / 2 (see below)
            b[j] = 0.5f * be;
          }
        }
        for (int y = ra - 1; y <= rb; ++y, ++seq) {
          const uint32_t slot = seq % kNS;
          mbar_wait(full_bar(slot), (seq / kNS) & 1u);
          if (y >= 0 && y < p.H) {
            // rows r of the strip <-> pixels x = w0 - 1 + r; only [rlo, rhi) lie inside the image.  r advances by 8, so the
            // swizzle term (r & 7) == r0 is constant and the granule address advances by 1024 B.
            const int rlo = w0 > 0 ? 0 : 1 - w0;
            const int rhi = min(kStripPx, p.W - w0 + 1);
            int r = r0 < rlo ? r0 + (((rlo - r0) + 7) & ~7) : r0;
            uint8_t* gp8 = gbase + kWBytes + slot * kStripBytes + r * 128 + ((q ^ r0) << 4);
#pragma unroll 4
            for (; r < rhi; r += 8, gp8 += 1024) {
              uint4* gp = reinterpret_cast<uint4*>(gp8);
              const uint4 v = *gp;
              const uint32_t xw[4] = {v.x, v.y, v.z, v.w};
              float o[8];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                // silu(z) = h + h tanh(h), h = z / 2 = fma(a / 2, x, b / 2) (exact scaling): 3 instructions per element
                const float h0 = fmaf(a[2 * e], __uint_as_float(xw[e] << 16), b[2 * e]);
                const float h1 = fmaf(a[2 * e + 1], __uint_as_float(xw[e] & 0xffff0000u), b[2 * e + 1]);
                float t0, t1;
                asm("tanh.approx.f32 %0, %1;" : "=f"(t0) : "f"(h0));
                asm("tanh.approx.f32 %0, %1;" : "=f"(t1) : "f"(h1));
                o[2 * e] = fmaf(h0, t0, h0);
                o[2 * e + 1] = fmaf(h1, t1, h1);
              }
              uint4 w4;
              w4.x = fd_pack_bf16(o[0], o[1]);
              w4.y = fd_pack_bf16(o[2], o[3]);
              w4.z = fd_pack_bf16(o[4], o[5]);
              w4.w = fd_pack_bf16(o[6], o[7]);
              *gp = w4;
            }
          }
          fence_proxy_async_smem();       // generic-proxy writes -> visible to tcgen05.cp (async proxy)
          mbar_arrive(xfull_bar(slot));
        }
      }
    }
  } else if (warp >= 2 && warp < 2 + kEpiWarps) {
    // ===================== epilogue =====================
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
    ec.H = p.H; ec.W = p.W; ec.Cout = kC; ec.Wt = kTileW;
    ec.shuffle_cq = 0;
    ec.tempty_remote = 0;
    ec.dbg = kDiag ? p.dbg : 0;
    ec.rt_stats = nullptr; ec.rt_gamma = nullptr; ec.rt_beta = nullptr; ec.rt_eps = 0.f; ec.s_rt = nullptr;
    ec.phase = -1;
    ec.head_out = nullptr; ec.head_w = nullptr; ec.head_b = nullptr; ec.head_n = 0; ec.s_head = nullptr;
    ec.head_h0 = ec.head_w0 = ec.head_pt = ec.head_pl = 0;
    StripWalk walk(p);
    int j = 0, n = 0, w0 = 0, ra = 0, rb = 0;
    auto next = [&](int, EpiTile& t) {
      while (ra + j >= rb) {
        if (!walk.next(p, n, w0, ra, rb)) return false;
        j = 0;
      }
      t.img = n;
      t.h0 = ra + j;
      t.w0 = w0;
      t.n_tile = 0;
      ++j;
      return true;
    };
    strip_epilogue2<GPT>(ec, next);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace

// (C0, C1) in {(64, 0), (64, 64), (128, 0)}; Cout = 64; 3x3, pad 1
struct StripInputNorm {           // fused GroupNorm + SiLU on the input (null stats = none)
  const double* stats;
  const float *gamma, *beta, *scale_shift;
  long ss_stride;
  float eps;
};

static int strip_launch(const void* src0, int C0, const void* src1, int C1, const void* wpacked, const float* bias,
                        const void* residual, void* out, double* gn_stats, int N, int H, int W, const StripInputNorm& in,
                        cudaStream_t st);

int fd_conv3x3_strip_launch(const void* src0, int C0, const void* src1, int C1, const void* wpacked, const float* bias,
                            const void* residual, void* out, double* gn_stats, int N, int H, int W, cudaStream_t st) {
  return strip_launch(src0, C0, src1, C1, wpacked, bias, residual, out, gn_stats, N, H, W, StripInputNorm{}, st);
}

extern "C" int fd_conv3x3_gnsilu_in(const void* src, const double* in_stats, const float* in_gamma, const float* in_beta,
                                    const float* in_scale_shift, long in_ss_stride, float in_eps, const void* wpacked,
                                    const float* bias, const void* residual, void* out, double* gn_stats, int N, int H, int W,
                                    void* stream) {
  FD_REQUIRE(src && in_stats && in_gamma && in_beta && wpacked && out && N > 0 && H > 0 && W >= 64,
             "conv3x3_gnsilu_in: bad argument (needs 64 -> 64 channels, W >= 64)");
  StripInputNorm in{in_stats, in_gamma, in_beta, in_scale_shift, in_ss_stride, in_eps};
  return strip_launch(src, 64, nullptr, 0, wpacked, bias, residual, out, gn_stats, N, H, W, in, (cudaStream_t)stream);
}

static int strip_launch(const void* src0, int C0, const void* src1, int C1, const void* wpacked, const float* bias,
                        const void* residual, void* out, double* gn_stats, int N, int H, int W, const StripInputNorm& in,
                        cudaStream_t st) {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    FD_CUDA(cudaGetDevice(&dev));
    FD_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  }
  const int cin = C0 + C1;
  const int passes = cin / 64;
  StripParams p{};
  p.N = N; p.H = H; p.W = W;
  p.tile_w = kTileW;
  p.wblocks = (W + p.tile_w - 1) / p.tile_w;
  p.total_rows = N * p.wblocks * H;
  p.w_kstride = cin;
  CUtensorMap mw, mo;
  {
    const uint64_t dO[5] = {(uint64_t)kC, (uint64_t)W, (uint64_t)H, (uint64_t)N, 1};
    const uint64_t sO[4] = {(uint64_t)kC * 2, (uint64_t)W * kC * 2, (uint64_t)H * W * kC * 2, (uint64_t)N * H * W * kC * 2};
    const uint32_t box_out[5] = {64, (uint32_t)p.tile_w, 1, 1, 1};
    if (int e = make_tmap_bf16(&mo, out, 5, dO, sO, box_out)) return e;
    const uint64_t K = (uint64_t)9 * cin;
    const uint64_t dims[2] = {K, (uint64_t)kC};
    const uint64_t str[1] = {K * 2};
    const uint32_t box[2] = {64, 64};
    if (int e = make_tmap_bf16(&mw, wpacked, 2, dims, str, box)) return e;
  }
  const int grid = p.total_rows < sms ? p.total_rows : sms;
  static bool attr_set = false;
  if (!attr_set) {
    FD_CUDA(cudaFuncSetAttribute(conv3x3_strip_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    FD_CUDA(cudaFuncSetAttribute(conv3x3_strip_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    attr_set = true;
  }
  // A operand from tensor memory.  Measured at 8x440x1024: 64->64 0.214 ms against 0.226 for the former shared-memory-operand
  // (SS) issuer, 128->64 0.510 against 0.535; the outputs were bit-identical.  With the operand reads gone the layer is held by
  // the single issuing thread (it runs only 2-3 MMAs ahead of the pipe) and by its HBM traffic (922 MB = 0.141 ms at the copy
  // peak, 0.175 ms measured with MMAs and copies disabled).  An L2 prefetch of the input rows ahead of their TMA loads was
  // measured no faster (0.229 -> 0.231 ms).
  p.in_stats = in.stats;
  p.in_gamma = in.gamma;
  p.in_beta = in.beta;
  p.in_ss = in.scale_shift;
  p.in_ss_stride = in.ss_stride;
  p.in_eps = in.eps;
  static const int dbg = fd_diag_bits("FD_CONV_DBG");
  p.dbg = dbg;
  for (int pass = 0; pass < passes; ++pass) {
    const bool last = pass == passes - 1;
    const bool from1 = pass == 1 && C1 > 0;                 // second half comes from the second tensor
    const void* src = from1 ? src1 : src0;
    const int csrc = from1 ? C1 : C0;
    CUtensorMap mi;
    const uint64_t d[5] = {(uint64_t)csrc, (uint64_t)W, (uint64_t)H, (uint64_t)N, 1};
    const uint64_t sB[4] = {(uint64_t)csrc * 2, (uint64_t)W * csrc * 2, (uint64_t)H * W * csrc * 2, (uint64_t)N * H * W * csrc * 2};
    const uint32_t box_in[5] = {64, (uint32_t)kStripPx, 1, 1, 1};
    if (int e = make_tmap_bf16(&mi, src, 5, d, sB, box_in)) return e;
    p.c_off = (pass == 1 && C1 == 0) ? 64 : 0;
    p.w_k0 = pass * 64;
    p.bias = last ? bias : nullptr;
    // pass 0 adds the caller's residual (if any), pass 1 the partial sum of pass 0
    p.residual = static_cast<const __nv_bfloat16*>(pass > 0 ? out : residual);
    p.gn_stats = last ? gn_stats : nullptr;
    if (p.gn_stats != nullptr) conv3x3_strip_kernel<8><<<grid, kThreads, kSmemBytes, st>>>(mi, mw, mo, p);
    else conv3x3_strip_kernel<0><<<grid, kThreads, kSmemBytes, st>>>(mi, mw, mo, p);
    FD_LAUNCH_CHECK();
  }
  return FD_OK;
}
