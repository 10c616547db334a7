// Backward bilinear warp (warp.py:95-119) and the fused warp + Charbonnier photometric + end-point-error forward
// (losses.py:3-6,46-47) with the sampled frame staged in shared memory by TMA -- the forward kernels of BASELINE config #4.
//
// Why: the config's flow is white noise (sigma = 4 px), so the 12 bilinear taps of a pixel land in 12 different 32-byte
// sectors and a warp-wide gather instruction touches ~24 sectors in ~5.5 L1 wavefronts (ncu, profiles/r2_prof_warp_summary.txt:
// the one-thread-per-pixel kernels of fd_warp.cu sit at 65-73 % of the L1 data-pipe peak and move 3.9x the DRAM bytes from
// L2 to L1).  Shared memory has no sectors: a random 4-byte gather costs its bank conflicts (~3.4 wavefronts per warp
// instruction for 32 random banks) and nothing else, and the fill is one asynchronous bulk copy.
//
//   * persistent blocks (one per SM) walk 16 x 128 pixel tiles; for each tile ONE 3-d TMA load brings the
//     (16 + 2R + 1) x (128 + 2R + 4) window (R = 16 px = 4 sigma) of all three planes of the sampled frame into one of two
//     96 KB shared-memory buffers -- out-of-image parts arrive as zeros, which is exactly grid_sample's zero padding;
//   * the load of tile i + 1 is in flight while tile i is computed; the thread's own flow / target / frame1 values of tile
//     i + 1 are prefetched into registers at the same time, so a tile never waits for DRAM;
//   * a thread owns two consecutive pixels of a tile row (1024 threads per block); taps that fall outside the window (|flow| > 16 px: 6e-5 of the
//     taps of the config) take the global-memory path of fd_warp.cu with the reference's validity tests.
// Geometry, weights and the accumulation order are fd_warp_common.cuh's (the reference's op sequence), so `out` / `mask` stay
// bit-identical to fd_warp.cu and to the reference.  Three-channel frames with W % 4 == 0 only (else fd_warp.cu runs).
#include <cuda.h>
#include <atomic>

#include "fd_tc.cuh"
#include "fd_warp_common.cuh"

using namespace fdwarp;
using namespace fdtc;

namespace {

constexpr int kTH = 16, kTW = 128, kR = 16, kC = 3;
constexpr int kWH = kTH + 2 * kR + 1;            // 49 window rows: the south taps reach one row below the cell
constexpr int kWW = kTW + 2 * kR + 4;            // 164 window columns (16-byte multiple; east taps reach one column further)
constexpr int kWin = kWH * kWW;                  // floats per plane window
constexpr int kBufBytes = ((kC * kWin * 4 + 127) / 128) * 128;
constexpr int kTxBytes = kC * kWin * 4;          // bytes one TMA box delivers (out-of-bounds parts count)
#ifndef FD_WIN_PX
#define FD_WIN_PX 4
#endif
constexpr int kPx = FD_WIN_PX;                   // consecutive pixels per thread
constexpr int kThreads = kTH * kTW / kPx;        // 1024: 16 rows x 64 pairs (32 warps hide the division / gather latencies)
constexpr int kSmemBytes = 2 * kBufBytes + 128 /*barriers*/ + 128 /*alignment slack*/;

struct WinParams {
  const float* frame1;     // MODE 1
  const float* frame2;     // the sampled frame (global fallback path)
  const float* flow;
  const float* flow_gt;    // MODE 1
  float* out;              // MODE 0
  float* mask;             // MODE 0 (may be null)
  float* partials;         // MODE 1: [grid][3] floats, then (8-byte aligned) one 64-bit ticket word {launch tag, count}
  unsigned tag;            // MODE 1: this launch's non-zero tag (see the ticket protocol at the end of the kernel)
  float* sums;             // MODE 1: {photo sum, mask sum, EPE sum, pixel count}, written by the last block to finish
  // backward modes (2: plain warp given gout, 3: fused photometric + EPE objective given the forward sums)
  const float* gout;       // MODE 2
  const float* fsums;      // MODE 3: forward sums
  float g_photo, g_epe;    // MODE 3
  float* gflow;            // may be null (MODE 2)
  float* acc;              // (B, H, W, 4) pixel-interleaved gradient of the sampled frame, zeroed by the host; may be null
  BwGeom g;
  int B, tiles_x, tiles_y, ntiles;
  int dbg;                 // FD_WARP_WIN_DBG in FD_DIAG builds: 1 = no compute, 2 = no TMA (timing isolation only: wrong results)
};

template <int N> struct VecT;
template <> struct VecT<2> { using type = float2; };
template <> struct VecT<4> { using type = float4; };
using PxVec = VecT<kPx>::type;
__device__ __forceinline__ void unpack(const float2& v, float (&o)[2]) { o[0] = v.x; o[1] = v.y; }
[[maybe_unused]] __device__ __forceinline__ void unpack(const float4& v, float (&o)[4]) { o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; }
__device__ __forceinline__ float2 pack(const float (&o)[2]) { return make_float2(o[0], o[1]); }
[[maybe_unused]] __device__ __forceinline__ float4 pack(const float (&o)[4]) { return make_float4(o[0], o[1], o[2], o[3]); }

struct TileAt {
  int b, y0, x0;
};
__device__ __forceinline__ TileAt tile_at(unsigned t, unsigned tiles_x, unsigned tiles_y) {      // once per tile, unsigned
  TileAt r;
  const unsigned row = t / tiles_x, b = row / tiles_y;
  r.x0 = (int)((t - row * tiles_x) * kTW);
  r.b = (int)b;
  r.y0 = (int)((row - b * tiles_y) * kTH);
  return r;
}
__device__ __forceinline__ float rsqrt_approx(float x) {      // one MUFU.RSQ (rsqrtf adds a denormal-range fix-up; x >= 1e-6 here)
  float y;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {      // explicit shared-space load (a generic pointer would compile to LD)
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}

// MODE 0: out / mask.  MODE 1: photometric + EPE partial sums.  MODE 2 / 3: their backward passes (see WinParams).
template <int MODE>
__global__ void __launch_bounds__(kThreads, 1) warp_win_fwd_kernel(const __grid_constant__ CUtensorMap map_f2, const WinParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~(uintptr_t)127);
  const uint32_t win0 = smem_u32(base);               // two window buffers, kBufBytes apart
  const uint32_t bar0 = win0 + 2 * kBufBytes;
  __shared__ float red[3 * 32];
  const int tid = threadIdx.x;
  const BwGeom g = p.g;
  const BwDiv dv = bw_divisors(g);
  const int H = g.H, W = g.W;
  const long HW = (long)H * W;
  if (tid == 0) {
    tma_prefetch_desc(&map_f2);
    mbar_init(bar0, 1);
    mbar_init(bar0 + 8, 1);
    mbar_init(bar0 + 16, kThreads);      // "buffer 0 / 1 has been read by every thread" (no block barrier per tile: the warps
    mbar_init(bar0 + 24, kThreads);      //  drift up to one tile apart, only the issuing thread waits)
    fence_barrier_init();
  }
  __syncthreads();
  constexpr int kGroups = kTW / kPx;                 // pixel groups per tile row
  const int ry = tid / kGroups, cx = (tid % kGroups) * kPx;       // the thread's row / first column inside a tile

  auto issue = [&](const TileAt& a, int buf) {        // thread 0 only
    mbar_expect_tx(bar0 + 8 * buf, kTxBytes);
    tma_load_3d(win0 + buf * kBufBytes, &map_f2, bar0 + 8 * buf, a.x0 - kR, a.y0 - kR, a.b * kC);
  };
  // the thread's own streamed values of a tile: flow (dy, dx), and for MODE 1 the target flow and frame1
  struct Own {
    PxVec f0, f1, g0, g1, a[kC];
    bool exists;
  };
  auto load_own = [&](const TileAt& a, Own& o) {
    const int y = a.y0 + ry, x = a.x0 + cx;
    o.exists = y < H && x < W;                        // (W % 4 == 0: a pixel group is whole or absent)
    if (!o.exists) return;
    const long fo = (long)a.b * 2 * HW + (long)y * W + x;
    o.f0 = __ldg(reinterpret_cast<const PxVec*>(p.flow + fo));
    o.f1 = __ldg(reinterpret_cast<const PxVec*>(p.flow + fo + HW));
    if (MODE == 1 || MODE == 3) {
      o.g0 = __ldg(reinterpret_cast<const PxVec*>(p.flow_gt + fo));
      o.g1 = __ldg(reinterpret_cast<const PxVec*>(p.flow_gt + fo + HW));
    }
    if (MODE != 0) {
      const float* src = MODE == 2 ? p.gout : p.frame1;
      const long po = (long)a.b * kC * HW + (long)y * W + x;
#pragma unroll
      for (int c = 0; c < kC; ++c) o.a[c] = __ldg(reinterpret_cast<const PxVec*>(src + po + c * HW));
    }
  };
  float kp = 0.f, ke = 0.f;
  if (MODE == 3) {
    kp = p.g_photo / __ldg(p.fsums + 1);
    ke = p.g_epe / __ldg(p.fsums + 3);
  }

  float s[3] = {0.f, 0.f, 0.f};
  int tile = blockIdx.x;
  Own nxt;
  nxt.exists = false;
  TileAt ta_next = tile_at(tile < p.ntiles ? tile : 0, p.tiles_x, p.tiles_y);
  // tile += gridDim.x as a mixed-radix addition on (tile column, tile row, image): the two divisions per tile of tile_at
  // were 4 % of the instruction stream
  const unsigned g1 = gridDim.x / p.tiles_x;
  const int step_x = (int)(gridDim.x - g1 * p.tiles_x) * kTW, step_b = (int)(g1 / p.tiles_y);
  const int step_y = (int)(g1 - (unsigned)step_b * p.tiles_y) * kTH;
  const int lim_x = p.tiles_x * kTW, lim_y = p.tiles_y * kTH;
  if (tile < p.ntiles) {
    if (tid == 0 && !(kDiag && (p.dbg & 2))) issue(ta_next, 0);
    load_own(ta_next, nxt);
  }
  for (int it = 0; tile < p.ntiles; ++it, tile += gridDim.x) {
    const int buf = it & 1;
    const int next = tile + gridDim.x;
    const Own cur = nxt;
    const TileAt a = ta_next;
    if (next < p.ntiles) {
      ta_next.x0 += step_x;
      const int cx1 = ta_next.x0 >= lim_x;
      ta_next.x0 -= cx1 * lim_x;
      ta_next.y0 += step_y + cx1 * kTH;
      const int cy1 = ta_next.y0 >= lim_y;
      ta_next.y0 -= cy1 * lim_y;
      ta_next.b += step_b + cy1;
      if (tid == 0 && !(kDiag && (p.dbg & 2))) {
        // buffer buf ^ 1 was last read by tile it - 1: its (it - 1) / 2-th use
        if (it > 0) mbar_wait(bar0 + 16 + 8 * (buf ^ 1), (uint32_t)((it - 1) >> 1) & 1u);
        issue(ta_next, buf ^ 1);
      }
      load_own(ta_next, nxt);
    }
    if (!(kDiag && (p.dbg & 2))) mbar_wait(bar0 + 8 * buf, (uint32_t)(it >> 1) & 1u);
    if (cur.exists && !(kDiag && (p.dbg & 1))) {
      const int y = a.y0 + ry, x = a.x0 + cx;
      const int wy0 = a.y0 - kR, wx0 = a.x0 - kR;
      const uint32_t w0 = win0 + buf * kBufBytes;
      float fdy[kPx], fdx[kPx];
      unpack(cur.f0, fdy);
      unpack(cur.f1, fdx);
      if (MODE >= 2) {
        // ---- backward: gradient of the flow (gather) and of the sampled frame (one 128-bit reduction per tap into the
        // pixel-interleaved buffer: the three channels of a tap share their address) ----
        float av[kC][kPx];
#pragma unroll
        for (int c = 0; c < kC; ++c) unpack(cur.a[c], av[c]);
        float gxo[kPx], gyo[kPx];
#pragma unroll
        for (int j = 0; j < kPx; ++j) {
          BwTaps t;
          bw_taps(fdx[j], fdy[j], x + j, y, g, dv, t);
          const float mj = MODE == 3 ? bw_mask_fast(t) : 1.f;
          const int wy = t.y0 - wy0, wx = t.x0 - wx0;
          const bool inwin = wy >= 0 && wy + 1 < kWH && wx >= 0 && wx + 1 < kWW && (t.okx0 || t.okx1) && (t.oky0 || t.oky1);
          const uint32_t q = w0 + (uint32_t)(wy * kWW + wx) * 4u;
          float gw[kC], dix = 0.f, diy = 0.f;
#pragma unroll
          for (int c = 0; c < kC; ++c) {
            BwVals v;
            if (inwin) {
              v.nw = lds_f32(q + (c * kWin) * 4);
              v.ne = lds_f32(q + (c * kWin + 1) * 4);
              v.sw = lds_f32(q + (c * kWin + kWW) * 4);
              v.se = lds_f32(q + (c * kWin + kWW + 1) * 4);
            } else {
              v = bw_gather(p.frame2 + ((long)a.b * kC + c) * HW, t, W);
            }
            if (MODE == 3) {
              const float d = av[c][j] - bw_sample(v, t);
              gw[c] = -kp * mj * d * rsqrt_approx(d * d + 1e-6f);      // dL/dwarped; one MUFU (2 ulp) for 1 / sqrt
            } else {
              gw[c] = av[c][j];
            }
            dix += gw[c] * ((v.ne - v.nw) * t.sy + (v.se - v.sw) * t.ny);
            diy += gw[c] * ((v.sw - v.nw) * t.ex + (v.se - v.ne) * t.wx);
          }
          gxo[j] = bw_div_rn(dix * g.half_w, dv.w) * 2.f;
          gyo[j] = bw_div_rn(diy * g.half_h, dv.h) * 2.f;
          if (p.acc != nullptr && (MODE == 2 || gw[0] != 0.f || gw[1] != 0.f || gw[2] != 0.f)) {
            float* cell = p.acc + (((long)a.b * H + t.y0) * W + t.x0) * 4;
            auto red4 = [&](float* dst, float wt) {
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(gw[0] * wt), "f"(gw[1] * wt),
                           "f"(gw[2] * wt), "f"(0.f)
                           : "memory");
            };
            if (t.okx0 && t.oky0) red4(cell, t.nw);
            if (t.okx1 && t.oky0) red4(cell + 4, t.ne);
            if (t.okx0 && t.oky1) red4(cell + (long)W * 4, t.sw);
            if (t.okx1 && t.oky1) red4(cell + (long)W * 4 + 4, t.se);
          }
        }
        if (p.gflow != nullptr) {
          if (MODE == 3) {
            float gdy[kPx], gdx[kPx];
            unpack(cur.g0, gdy);
            unpack(cur.g1, gdx);
#pragma unroll
            for (int j = 0; j < kPx; ++j) {
              const float du = fdy[j] - gdy[j], dvv = fdx[j] - gdx[j];
              const float n2 = du * du + dvv * dvv;
              const float inv = n2 > 0.f ? ke * rsqrt_approx(n2) : 0.f;
              gyo[j] += du * inv;
              gxo[j] += dvv * inv;
            }
          }
          const long fo = (long)a.b * 2 * HW + (long)y * W + x;
          *reinterpret_cast<PxVec*>(p.gflow + fo) = pack(gyo);
          *reinterpret_cast<PxVec*>(p.gflow + fo + HW) = pack(gxo);
        }
      } else {
      float o[kC][kPx], m[kPx];
#pragma unroll
      for (int j = 0; j < kPx; ++j) {
        BwTaps t;
        bw_taps(fdx[j], fdy[j], x + j, y, g, dv, t);
        m[j] = bw_mask_fast(t);
        const int wy = t.y0 - wy0, wx = t.x0 - wx0;
        // A cell with no valid column (row) was clamped to column (row) 0 by bw_taps -- all of its taps are invalid although
        // the clamped address holds image data: such cells (far outside the image) take the checked global path.  For every
        // other in-window cell the zero padding that came with the copy IS the validity test: taps outside the image read 0.
        const bool inwin = wy >= 0 && wy + 1 < kWH && wx >= 0 && wx + 1 < kWW && (t.okx0 || t.okx1) && (t.oky0 || t.oky1);
        if (inwin) {
          const uint32_t q = w0 + (uint32_t)(wy * kWW + wx) * 4u;
#pragma unroll
          for (int c = 0; c < kC; ++c) {
            BwVals v;
            v.nw = lds_f32(q + (c * kWin) * 4);
            v.ne = lds_f32(q + (c * kWin + 1) * 4);
            v.sw = lds_f32(q + (c * kWin + kWW) * 4);
            v.se = lds_f32(q + (c * kWin + kWW + 1) * 4);
            o[c][j] = bw_sample(v, t);
          }
        } else {
#pragma unroll
          for (int c = 0; c < kC; ++c) o[c][j] = bw_sample(bw_gather(p.frame2 + ((long)a.b * kC + c) * HW, t, W), t);
        }
      }
      if (MODE == 0) {
        const long po = (long)a.b * kC * HW + (long)y * W + x;
#pragma unroll
        for (int c = 0; c < kC; ++c) {
          *reinterpret_cast<PxVec*>(p.out + po + c * HW) = pack(o[c]);
          if (p.mask != nullptr) *reinterpret_cast<PxVec*>(p.mask + po + c * HW) = pack(m);
        }
      } else {
        float gdy[kPx], gdx[kPx];
        unpack(cur.g0, gdy);
        unpack(cur.g1, gdx);
#pragma unroll
        for (int j = 0; j < kPx; ++j) {
          const float du = fdy[j] - gdy[j], dv = fdx[j] - gdx[j];
          const float e2 = du * du + dv * dv;
          s[2] += e2 > 0.f ? e2 * rsqrt_approx(e2) : 0.f;      // (ftz: |d| < 1e-19 px counts as 0)
        }
#pragma unroll
        for (int c = 0; c < kC; ++c) {
          float av[kPx];
          unpack(cur.a[c], av);
#pragma unroll
          for (int j = 0; j < kPx; ++j) {
            const float d = av[j] - o[c][j];
            const float q2 = d * d + 1e-6f;
            s[0] += m[j] * (q2 * rsqrt_approx(q2));     // sqrt(q2), q2 >= 1e-6 (as fd_warp.cu)
            s[1] += m[j];
          }
        }
      }
      }   // forward modes
    }
    mbar_arrive(bar0 + 16 + 8 * buf);      // this thread's reads of win[buf] are done
  }
  if (MODE == 1) {
    fd_block_sum<3>(s, red);
    __shared__ int s_last;
    // Ticket = {tag of the launch that owns the count, number of blocks that have arrived}.  A block that finds another tag
    // (uninitialised workspace, or the leftovers of an aborted launch) starts the count at 1; the last block clears the word,
    // so that a replay of the SAME launch (a CUDA graph bakes the tag) starts clean as well.  The host therefore needs no
    // memset node in front of the kernel (it was ~5 us of a 47 us operation when the kernel is timed on its own).
    unsigned long long* ticket = reinterpret_cast<unsigned long long*>(
        (reinterpret_cast<uintptr_t>(p.partials + (size_t)gridDim.x * 3) + 7) & ~(uintptr_t)7);
    if (tid == 0) {
      p.partials[blockIdx.x * 3 + 0] = s[0];
      p.partials[blockIdx.x * 3 + 1] = s[1];
      p.partials[blockIdx.x * 3 + 2] = s[2];
      __threadfence();
      // One compare-and-swap from the clean state for the first block, one fetch-add for everybody else (a compare-and-swap
      // retry loop for all 148 blocks, which arrive together, serialises into ~148 L2 round trips: measured +47 us).
      const unsigned long long first = ((unsigned long long)p.tag << 32) | 1ull;
      unsigned long long expect = 0ull, neu;
      for (;;) {
        const unsigned long long prev = atomicCAS(ticket, expect, first);
        if (prev == expect) {
          neu = first;
          break;
        }
        if ((unsigned)(prev >> 32) == p.tag) {          // this launch owns the word: nobody replaces it before we have arrived
          neu = atomicAdd(ticket, 1ull) + 1ull;
          break;
        }
        expect = prev;                                  // a foreign word: replace exactly that
      }
      s_last = (unsigned)neu == gridDim.x;
    }
    __syncthreads();
    // The last block to finish reduces the per-block partials in a FIXED order in double precision (deterministic whatever
    // the block completion order), which saves the separate one-block finalize launch (~7 us of a ~50 us operation).
    if (s_last && tid < 32) {
      __threadfence();
      double acc[3] = {0.0, 0.0, 0.0};
      for (unsigned k = tid; k < gridDim.x; k += 32) {
        const volatile float* q = p.partials + (size_t)k * 3;
        acc[0] += (double)q[0];
        acc[1] += (double)q[1];
        acc[2] += (double)q[2];
      }
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
      if (tid == 0) {
        p.sums[0] = (float)acc[0];
        p.sums[1] = (float)acc[1];
        p.sums[2] = (float)acc[2];
        p.sums[3] = (float)((double)p.B * H * W);
        *ticket = 0ull;                        // every block of this launch has arrived: nobody touches the word any more
      }
    }
  }
}

// pixel-interleaved gradient (B, H, W, 4) -> planar (B, 3, H, W)
__global__ void __launch_bounds__(256) acc_to_planes3_kernel(const float* __restrict__ acc, float* __restrict__ g, int B, long HW) {
  const long total = (long)B * HW;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long b = i / HW, p = i - b * HW;
    const float4 a = __ldg(reinterpret_cast<const float4*>(acc) + i);
    g[(b * 3 + 0) * HW + p] = a.x;
    g[(b * 3 + 1) * HW + p] = a.y;
    g[(b * 3 + 2) * HW + p] = a.z;
  }
}

}  // namespace

int fd_warp_win_grid(int B, int H, int W) {
  const long tiles = (long)B * ((H + kTH - 1) / kTH) * ((W + kTW - 1) / kTW);
  return (int)(tiles < FD_NUM_SMS ? tiles : FD_NUM_SMS);
}

// Backward passes on the forward kernel's skeleton (same TMA windows for the gathers): mode 2 = plain warp given gout, mode 3 =
// fused photometric + EPE objective.  The gradient of the sampled frame is accumulated in `acc` (B, H, W, 4 floats, 16-byte
// aligned workspace) with one 128-bit reduction per tap and converted to the planar `gimage` by a second launch.
int fd_warp_bwd_win2(int mode, const float* frame1, const float* frame2, const float* flow, const float* flow_gt, const float* gout,
                     const float* fsums, float g_photo, float g_epe, float* gflow, float* gimage, float* acc, int B, int H, int W,
                     cudaStream_t st) {
  FD_REQUIRE(W % 4 == 0 && (mode == 2 || mode == 3), "warp_win_bwd2: bad argument");
  FD_REQUIRE(gimage == nullptr || (acc != nullptr && (reinterpret_cast<uintptr_t>(acc) & 15) == 0), "warp_win_bwd2: workspace");
  WinParams p{};
  p.frame1 = frame1; p.frame2 = frame2; p.flow = flow; p.flow_gt = flow_gt; p.gout = gout; p.fsums = fsums;
  p.g_photo = g_photo; p.g_epe = g_epe; p.gflow = gflow; p.acc = gimage != nullptr ? acc : nullptr;
  p.g = make_geom(H, W);
  p.B = B;
  p.tiles_x = (W + kTW - 1) / kTW;
  p.tiles_y = (H + kTH - 1) / kTH;
  const long tiles = (long)B * p.tiles_x * p.tiles_y;
  FD_REQUIRE(tiles < (1L << 31), "warp_win_bwd2: too many tiles");
  p.ntiles = (int)tiles;
  CUtensorMap map;
  {
    const uint64_t dims[3] = {(uint64_t)W, (uint64_t)H, (uint64_t)B * kC};
    const uint64_t str[2] = {(uint64_t)W * 4, (uint64_t)H * W * 4};
    const uint32_t box[3] = {(uint32_t)kWW, (uint32_t)kWH, (uint32_t)kC};
    if (int e = make_tmap_f32_plain(&map, frame2, 3, dims, str, box)) return e;
  }
  if (p.acc != nullptr) FD_CUDA(cudaMemsetAsync(acc, 0, sizeof(float) * 4 * (size_t)B * H * W, st));
  const int grid = fd_warp_win_grid(B, H, W);
  static bool attr_done[2] = {false, false};
  if (mode == 2) {
    if (!attr_done[0]) {
      FD_CUDA(cudaFuncSetAttribute(warp_win_fwd_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
      attr_done[0] = true;
    }
    warp_win_fwd_kernel<2><<<grid, kThreads, kSmemBytes, st>>>(map, p);
  } else {
    if (!attr_done[1]) {
      FD_CUDA(cudaFuncSetAttribute(warp_win_fwd_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
      attr_done[1] = true;
    }
    warp_win_fwd_kernel<3><<<grid, kThreads, kSmemBytes, st>>>(map, p);
  }
  FD_LAUNCH_CHECK();
  if (gimage != nullptr) {
    long blocks = ((long)B * H * W + 255) / 256;
    if (blocks > (long)FD_NUM_SMS * 16) blocks = (long)FD_NUM_SMS * 16;
    acc_to_planes3_kernel<<<(unsigned)blocks, 256, 0, st>>>(acc, gimage, B, (long)H * W);
    FD_LAUNCH_CHECK();
  }
  return FD_OK;
}

// mode 0: out / mask; mode 1: sums[4] = {photo sum, mask sum, EPE sum, pixel count}, partials = workspace of
// fd_warp_win_grid * 3 + 1 floats.  C == 3, W % 4 == 0.
int fd_warp_fwd_win(int mode, const float* frame1, const float* frame2, const float* flow, const float* flow_gt, float* out,
                    float* mask, float* partials, float* sums, int B, int H, int W, cudaStream_t st) {
  FD_REQUIRE(W % 4 == 0, "warp_win: W %% 4 != 0");
  FD_REQUIRE((reinterpret_cast<uintptr_t>(frame2) & 15) == 0 && (reinterpret_cast<uintptr_t>(flow) & 15) == 0,
             "warp_win: 16-byte aligned tensors");
  WinParams p{};
  p.frame1 = frame1; p.frame2 = frame2; p.flow = flow; p.flow_gt = flow_gt; p.out = out; p.mask = mask; p.partials = partials; p.sums = sums;
  p.g = make_geom(H, W);
  p.B = B;
  p.tiles_x = (W + kTW - 1) / kTW;
  p.tiles_y = (H + kTH - 1) / kTH;
  const long tiles = (long)B * p.tiles_x * p.tiles_y;
  FD_REQUIRE(tiles < (1L << 31), "warp_win: too many tiles");
  p.ntiles = (int)tiles;
  static const int dbg = fd_diag_bits("FD_WARP_WIN_DBG");
  p.dbg = dbg;
  CUtensorMap map;
  {
    const uint64_t dims[3] = {(uint64_t)W, (uint64_t)H, (uint64_t)B * kC};
    const uint64_t str[2] = {(uint64_t)W * 4, (uint64_t)H * W * 4};
    const uint32_t box[3] = {(uint32_t)kWW, (uint32_t)kWH, (uint32_t)kC};
    if (int e = make_tmap_f32_plain(&map, frame2, 3, dims, str, box)) return e;
  }
  const int grid = fd_warp_win_grid(B, H, W);
  static bool attr_done[2] = {false, false};
  if (mode == 0) {
    if (!attr_done[0]) {
      FD_CUDA(cudaFuncSetAttribute(warp_win_fwd_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
      attr_done[0] = true;
    }
    warp_win_fwd_kernel<0><<<grid, kThreads, kSmemBytes, st>>>(map, p);
  } else {
    if (!attr_done[1]) {
      FD_CUDA(cudaFuncSetAttribute(warp_win_fwd_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
      attr_done[1] = true;
    }
    static std::atomic<unsigned> next_tag{0};
    do {
      p.tag = ++next_tag;                      // unique per launch, never 0
    } while (p.tag == 0);
    warp_win_fwd_kernel<1><<<grid, kThreads, kSmemBytes, st>>>(map, p);
  }
  FD_LAUNCH_CHECK();
  return FD_OK;
}
