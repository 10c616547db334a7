// Backward of the bilinear warp (warp.py:95-119 under autograd) and of the fused warp + Charbonnier photometric + end-point-error
// objective (losses.py:3-6,46-47) with BOTH the sampled frame and its gradient staged in shared memory -- the backward
// kernels of BASELINE config #4.
//
// fd_warp.cu's backward gathers every tap through L1 (see fd_warp_win.cu for what white-noise flow does to that) and scatters
// the frame gradient with 12 red.global.add.f32 per pixel at random addresses (43 M scalar reductions per call).  Here a
// persistent block walks 16 x 128 pixel tiles channel by channel ("unit" = tile x channel):
//   * the (16 + 2R + 1) x (128 + 2R + 4) window (R = 16 px) of the frame plane arrives by one TMA load (zero padded),
//     two units ahead of its use;
//   * the gradient of that window is accumulated in shared memory (red.shared.add.f32: no sectors, no L2 round trips) and
//     leaves as ONE TMA reduce-add (cp.reduce.async.bulk.tensor ... .add) per unit -- the out-of-image part of the window is
//     clipped by the tensor map, so the in-window path needs no validity tests at all; four accumulation windows rotate so
//     that a window is being reduced, one filled, one zeroed at any time, with ONE block barrier per unit;
//     (TMA reductions with a NEGATIVE box origin are an illegal instruction on this part -- scripts/micro/tma_reduce.cu --
//     so the windows of the tiles on the top / left image border, 16 % of them, are flushed by the threads instead, with
//     128-bit red.global.add.v4.f32 on their non-zero groups);
//   * a thread owns four consecutive pixels and keeps their taps (cell, two fractions, flags) in registers across the three
//     channel passes; its own flow / target / frame1 (or upstream gradient) values of the next tile are prefetched.
// Measured limits (profiles/r2_prof_warp_summary.txt): this part has NO native fp32 shared-memory add -- red.shared.add.f32
// compiles to a load / add / compare-and-swap loop per address (ATOMS.CAST.SPIN): 88 of the kernel's 640 instructions per
// pixel and its top stall (short scoreboard).  Interleaving the four loops of a tap group by hand (four CAS in flight) was
// slower still (304 vs 199 us: divergent retry loops).  So the gain over the global-atomic kernels is 15-18 %, not the 2x of
// the forward pass.
// Taps outside the window (|flow| > 16 px) and cells clamped by bw_taps take fd_warp.cu's checked global path (global atomics).
// Same formulas and operation order per pixel as fd_warp.cu; the frame gradient is a sum of the same terms in a different
// order (tests: tolerance of the atomics, as before).  Three-channel frames with W % 4 == 0 only.
#include <cuda.h>
#include "fd_tc.cuh"
#include "fd_warp_common.cuh"

using namespace fdwarp;
using namespace fdtc;

namespace {

constexpr int kTH = 16, kTW = 128, kR = 16, kC = 3, kPx = 4;
constexpr int kWH = kTH + 2 * kR + 1;            // 49
constexpr int kWW = kTW + 2 * kR + 4;            // 164
constexpr int kWin = kWH * kWW;                  // floats per plane window
constexpr int kWinBytes = ((kWin * 4 + 127) / 128) * 128;
constexpr int kTxBytes = kWin * 4;
constexpr int kThreads = kTH * kTW / kPx;        // 512
constexpr int kAcc = 4;                          // accumulation windows in rotation
constexpr int kFr = 3;                           // frame windows in rotation: loaded two units ahead of their use
constexpr int kSmemBytes = (kFr + kAcc) * kWinBytes + 128 /*barriers*/ + 128 /*alignment slack*/;

struct BwdParams {
  const float* frame1;     // MODE 1
  const float* frame2;     // the sampled frame / image
  const float* flow;
  const float* flow_gt;    // MODE 1
  const float* gout;       // MODE 0: upstream gradient of the warped image
  const float* sums;       // MODE 1: forward sums {photo, mask, epe, count}
  float g_photo, g_epe;    // MODE 1
  float* gflow;            // may be null (MODE 0)
  float* gimage;           // gradient of the sampled frame (zeroed by the host); may be null
  BwGeom g;
  int B, tiles_x, tiles_y, ntiles;
  int dbg;                 // FD_WARP_WIN_DBG in FD_DIAG builds (isolation runs, wrong results): 4 = no TMA reduction, 8 = no shared-memory scatter, 16 = no TMA loads, 64 = no zeroing / proxy fence
};

struct TileAt {
  int b, y0, x0;
};
__device__ __forceinline__ TileAt tile_at(unsigned t, unsigned tiles_x, unsigned tiles_y) {
  TileAt r;
  const unsigned row = t / tiles_x, b = row / tiles_y;
  r.x0 = (int)((t - row * tiles_x) * kTW);
  r.b = (int)b;
  r.y0 = (int)((row - b * tiles_y) * kTH);
  return r;
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ float rsqrt_approx(float x) {
  float y;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void reds_f32(uint32_t addr, float v) {
  asm volatile("red.shared.add.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void sts_zero4(uint32_t addr) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %1, %1, %1};" ::"r"(addr), "f"(0.f) : "memory");
}
__device__ __forceinline__ void tma_reduce_add_3d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(m),
               "r"(src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}

// MODE 0: backward of out = warp(image, flow) given gout.  MODE 1: backward of the fused photometric + EPE objective.
template <int MODE>
__global__ void __launch_bounds__(kThreads, 1) warp_win_bwd_kernel(const __grid_constant__ CUtensorMap map_in,
                                                                   const __grid_constant__ CUtensorMap map_grad, const BwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~(uintptr_t)127);
  const uint32_t frame0 = smem_u32(base);                       // kFr frame windows
  const uint32_t acc0 = frame0 + kFr * kWinBytes;                 // kAcc accumulation windows
  const uint32_t bar0 = acc0 + kAcc * kWinBytes;
  const int tid = threadIdx.x;
  const BwGeom g = p.g;
  const BwDiv dv = bw_divisors(g);
  const int H = g.H, W = g.W;
  const long HW = (long)H * W;
  const bool want_gi = p.gimage != nullptr, want_gf = p.gflow != nullptr;
  if (tid == 0) {
    tma_prefetch_desc(&map_in);
    tma_prefetch_desc(&map_grad);
    for (int i = 0; i < kFr; ++i) mbar_init(bar0 + 8 * i, 1);
    fence_barrier_init();
  }
  auto zero_acc = [&](int slot) {
    const uint32_t a = acc0 + slot * kWinBytes;
    for (int i = tid; i < kWin / 4; i += kThreads) sts_zero4(a + i * 16);
  };
  // window -> global plane by the threads (border tiles): one vector reduction per non-zero group of four inside the image
  auto flush_manual = [&](int slot, int ox, int oy, int plane) {
    const uint32_t a = acc0 + slot * kWinBytes;
    float* dst = p.gimage + (long)plane * HW;
    for (int i = tid; i < kWin / 4; i += kThreads) {
      const int r = i / (kWW / 4), c4 = i - r * (kWW / 4);
      const int gy = oy + r, gx = ox + c4 * 4;
      if (gy < 0 || gy >= H || gx < 0 || gx >= W) continue;
      float4 v;
      asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a + i * 16));
      if (v.x == 0.f && v.y == 0.f && v.z == 0.f && v.w == 0.f) continue;
      asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + (long)gy * W + gx), "f"(v.x), "f"(v.y), "f"(v.z),
                   "f"(v.w)
                   : "memory");
    }
  };
  if (want_gi) zero_acc(0);
  __syncthreads();
  const int ry = tid / (kTW / kPx), cx = (tid % (kTW / kPx)) * kPx;
  float kp = 0.f, ke = 0.f;
  if (MODE == 1) {
    kp = p.g_photo / __ldg(p.sums + 1);
    ke = p.g_epe / __ldg(p.sums + 3);
  }

  struct Own {
    float4 f0, f1, g0, g1, a[kC];      // flow (dy, dx); MODE 1: target flow, frame1; MODE 0: a = gout
    bool exists;
  };
  auto load_own = [&](const TileAt& a, Own& o) {
    const int y = a.y0 + ry, x = a.x0 + cx;
    o.exists = y < H && x < W;
    if (!o.exists) return;
    const long fo = (long)a.b * 2 * HW + (long)y * W + x;
    o.f0 = __ldg(reinterpret_cast<const float4*>(p.flow + fo));
    o.f1 = __ldg(reinterpret_cast<const float4*>(p.flow + fo + HW));
    if (MODE == 1) {
      o.g0 = __ldg(reinterpret_cast<const float4*>(p.flow_gt + fo));
      o.g1 = __ldg(reinterpret_cast<const float4*>(p.flow_gt + fo + HW));
    }
    const float* src = MODE == 1 ? p.frame1 : p.gout;
    const long po = (long)a.b * kC * HW + (long)y * W + x;
#pragma unroll
    for (int c = 0; c < kC; ++c) o.a[c] = __ldg(reinterpret_cast<const float4*>(src + po + c * HW));
  };
  auto issue_load = [&](const TileAt& a, int c, unsigned u) {      // thread 0: frame window of unit u
    if (kDiag && (p.dbg & 16)) return;
    const uint32_t bar = bar0 + 8 * (u % kFr);
    mbar_expect_tx(bar, kTxBytes);
    tma_load_3d(frame0 + (u % kFr) * kWinBytes, &map_in, bar, a.x0 - kR, a.y0 - kR, a.b * kC + c);
  };

  // tile += gridDim.x as a mixed-radix addition (see fd_warp_win.cu)
  const unsigned g1 = gridDim.x / p.tiles_x;
  const int step_x = (int)(gridDim.x - g1 * p.tiles_x) * kTW, step_b = (int)(g1 / p.tiles_y);
  const int step_y = (int)(g1 - (unsigned)step_b * p.tiles_y) * kTH;
  const int lim_x = p.tiles_x * kTW, lim_y = p.tiles_y * kTH;

  int tile = blockIdx.x;
  if (tile >= p.ntiles) return;
  TileAt ta = tile_at(tile, p.tiles_x, p.tiles_y), ta_next = ta;
  Own nxt;
  load_own(ta, nxt);
  if (tid == 0) {
    issue_load(ta, 0, 0);
    issue_load(ta, 1, 1);
  }
  unsigned u = 0;                 // unit counter of this block
  int pv_x = 0, pv_y = 0, pv_p = 0;      // window origin / plane of the previous unit (its reduction is issued one unit later)
  for (; tile < p.ntiles; tile += gridDim.x) {
    const Own cur = nxt;
    ta = ta_next;
    const bool has_next = tile + (int)gridDim.x < p.ntiles;
    const int y = ta.y0 + ry, x = ta.x0 + cx;
    const int wy0 = ta.y0 - kR, wx0 = ta.x0 - kR;
    // taps of the thread's four pixels, kept across the channel passes
    uint32_t cell[kPx];           // in window: byte offset of the cell inside a window; else unused
    float wx[kPx], ny[kPx], m[kPx], dix[kPx], diy[kPx];
    bool inw[kPx];
    float fdy[kPx] = {cur.f0.x, cur.f0.y, cur.f0.z, cur.f0.w}, fdx[kPx] = {cur.f1.x, cur.f1.y, cur.f1.z, cur.f1.w};
#pragma unroll
    for (int j = 0; j < kPx; ++j) {
      BwTaps t;
      bw_taps(fdx[j], fdy[j], x + j, y, g, dv, t);
      m[j] = MODE == 1 ? bw_mask_fast(t) : 1.f;
      const int wy = t.y0 - wy0, wxx = t.x0 - wx0;
      inw[j] = cur.exists && wy >= 0 && wy + 1 < kWH && wxx >= 0 && wxx + 1 < kWW && (t.okx0 || t.okx1) && (t.oky0 || t.oky1);
      cell[j] = (uint32_t)(wy * kWW + wxx) * 4u;
      wx[j] = t.wx;
      ny[j] = t.ny;
      dix[j] = diy[j] = 0.f;
    }
#pragma unroll 1
    for (int c = 0; c < kC; ++c, ++u) {
      __syncthreads();            // unit u - 1 is complete in shared memory: its scatters, its reads of frame slot (u - 1) % kFr
      const bool pv_manual = pv_x < 0 || pv_y < 0;      // (block-uniform)
      if (want_gi && u > 0 && pv_manual && !(kDiag && (p.dbg & 4))) flush_manual((int)((u - 1) % kAcc), pv_x, pv_y, pv_p);
      if (tid == 0) {
        if (want_gi && u > 0 && !(kDiag && (p.dbg & 4))) {
          if (!pv_manual) tma_reduce_add_3d(&map_grad, acc0 + ((u - 1) % kAcc) * kWinBytes, pv_x, pv_y, pv_p);
          tma_store_commit();            // (an empty group for a thread-flushed unit: keeps the group count per unit uniform)
          tma_store_wait_read<1>();      // the reduction of unit u - 2 has read its window: it may be zeroed during unit u + 1
        }
        // frame window of unit u + 2 into the slot unit u - 1 just released
        if (c == 0) issue_load(ta, 2, u + 2);
        else if (has_next) {
          TileAt n = ta;
          n.x0 += step_x;
          const int c1 = n.x0 >= lim_x;
          n.x0 -= c1 * lim_x;
          n.y0 += step_y + c1 * kTH;
          const int c2 = n.y0 >= lim_y;
          n.y0 -= c2 * lim_y;
          n.b += step_b + c2;
          issue_load(n, c - 1, u + 2);
        }
      }
      pv_x = wx0; pv_y = wy0; pv_p = ta.b * kC + c;
      if (c == 1 && has_next) {          // next tile's coordinates and own values (a whole unit ahead of their use)
        ta_next = ta;
        ta_next.x0 += step_x;
        const int c1 = ta_next.x0 >= lim_x;
        ta_next.x0 -= c1 * lim_x;
        ta_next.y0 += step_y + c1 * kTH;
        const int c2 = ta_next.y0 >= lim_y;
        ta_next.y0 -= c2 * lim_y;
        ta_next.b += step_b + c2;
        load_own(ta_next, nxt);
      }
      if (!(kDiag && (p.dbg & 16))) mbar_wait(bar0 + 8 * (u % kFr), (u / kFr) & 1u);
      const uint32_t fw = frame0 + (u % kFr) * kWinBytes, aw = acc0 + (u % kAcc) * kWinBytes;
      if (cur.exists) {
        const float4 ac = c == 0 ? cur.a[0] : (c == 1 ? cur.a[1] : cur.a[2]);      // (no dynamic indexing: registers)
        const float av[kPx] = {ac.x, ac.y, ac.z, ac.w};
#pragma unroll
        for (int j = 0; j < kPx; ++j) {
          const float ex = __fsub_rn(1.f, wx[j]), sy = __fsub_rn(1.f, ny[j]);
          const float wnw = __fmul_rn(sy, ex), wne = __fmul_rn(sy, wx[j]), wsw = __fmul_rn(ny[j], ex), wse = __fmul_rn(ny[j], wx[j]);
          BwVals v;
          if (inw[j]) {
            v.nw = lds_f32(fw + cell[j]);
            v.ne = lds_f32(fw + cell[j] + 4);
            v.sw = lds_f32(fw + cell[j] + kWW * 4);
            v.se = lds_f32(fw + cell[j] + kWW * 4 + 4);
          } else {        // rare: the taps are recomputed rather than kept (an array of them would live in local memory)
            BwTaps t;
            bw_taps(fdx[j], fdy[j], x + j, y, g, dv, t);
            v = bw_gather(p.frame2 + ((long)ta.b * kC + c) * HW, t, W);
          }
          float gw;
          if (MODE == 1) {
            float s = __fmul_rn(v.nw, wnw);
            s = __fmaf_rn(v.ne, wne, s);
            s = __fmaf_rn(v.sw, wsw, s);
            s = __fmaf_rn(v.se, wse, s);
            const float d = av[j] - s;
            gw = -kp * m[j] * d * rsqrt_approx(d * d + 1e-6f);   // dL/dwarped; one MUFU (2 ulp) instead of IEEE sqrt + division
          } else {
            gw = av[j];
          }
          if (want_gf || MODE == 1) {
            dix[j] += gw * ((v.ne - v.nw) * sy + (v.se - v.sw) * ny[j]);
            diy[j] += gw * ((v.sw - v.nw) * ex + (v.se - v.ne) * wx[j]);
          }
          if (want_gi && (MODE == 0 || gw != 0.f)) {
            if (inw[j] && kDiag && (p.dbg & 8)) {
            } else if (inw[j]) {
              reds_f32(aw + cell[j], gw * wnw);
              reds_f32(aw + cell[j] + 4, gw * wne);
              reds_f32(aw + cell[j] + kWW * 4, gw * wsw);
              reds_f32(aw + cell[j] + kWW * 4 + 4, gw * wse);
            } else {
              BwTaps t;
              bw_taps(fdx[j], fdy[j], x + j, y, g, dv, t);
              float* r0 = p.gimage + ((long)ta.b * kC + c) * HW + (long)t.y0 * W + t.x0;
              if (t.okx0 && t.oky0) atomicAdd(r0, gw * wnw);
              if (t.okx1 && t.oky0) atomicAdd(r0 + 1, gw * wne);
              if (t.okx0 && t.oky1) atomicAdd(r0 + W, gw * wsw);
              if (t.okx1 && t.oky1) atomicAdd(r0 + W + 1, gw * wse);
            }
          }
        }
      }
      if (want_gi && !(kDiag && (p.dbg & 64))) {
        zero_acc((int)((u + 1) % kAcc));       // last used by unit u - 3, whose reduction has finished reading (see above)
        fence_proxy_async_smem();              // this unit's red.shared results -> visible to the TMA reduction issued after the barrier
      }
    }
    if (want_gf && cur.exists) {
      float gy[kPx], gx[kPx];
#pragma unroll
      for (int j = 0; j < kPx; ++j) {
        gx[j] = bw_div_rn(dix[j] * g.half_w, dv.w) * 2.f;
        gy[j] = bw_div_rn(diy[j] * g.half_h, dv.h) * 2.f;
      }
      if (MODE == 1) {
        const float gdy[kPx] = {cur.g0.x, cur.g0.y, cur.g0.z, cur.g0.w}, gdx[kPx] = {cur.g1.x, cur.g1.y, cur.g1.z, cur.g1.w};
#pragma unroll
        for (int j = 0; j < kPx; ++j) {
          const float du = fdy[j] - gdy[j], dvv = fdx[j] - gdx[j];
          const float n2 = du * du + dvv * dvv;
          const float inv = n2 > 0.f ? ke * rsqrt_approx(n2) : 0.f;
          gy[j] += du * inv;
          gx[j] += dvv * inv;
        }
      }
      const long fo = (long)ta.b * 2 * HW + (long)y * W + x;
      *reinterpret_cast<float4*>(p.gflow + fo) = make_float4(gy[0], gy[1], gy[2], gy[3]);
      *reinterpret_cast<float4*>(p.gflow + fo + HW) = make_float4(gx[0], gx[1], gx[2], gx[3]);
    }
  }
  __syncthreads();
  if (want_gi && u > 0 && !(kDiag && (p.dbg & 4))) {
    const bool pv_manual = pv_x < 0 || pv_y < 0;
    if (pv_manual) flush_manual((int)((u - 1) % kAcc), pv_x, pv_y, pv_p);
    if (tid == 0) {
      if (!pv_manual) tma_reduce_add_3d(&map_grad, acc0 + ((u - 1) % kAcc) * kWinBytes, pv_x, pv_y, pv_p);
      tma_store_commit();
      tma_store_wait_all();
    }
  }
}

}  // namespace

// mode 0: gimage / gflow of the plain warp given gout; mode 1: gflow / gframe2 of the fused objective.  gimage zeroed by caller.
int fd_warp_bwd_win(int mode, const float* frame1, const float* frame2, const float* flow, const float* flow_gt, const float* gout,
                    const float* sums, float g_photo, float g_epe, float* gflow, float* gimage, int B, int H, int W, cudaStream_t st) {
  FD_REQUIRE(W % 4 == 0, "warp_win_bwd: W %% 4 != 0");
  BwdParams p{};
  p.frame1 = frame1; p.frame2 = frame2; p.flow = flow; p.flow_gt = flow_gt; p.gout = gout; p.sums = sums;
  p.g_photo = g_photo; p.g_epe = g_epe; p.gflow = gflow; p.gimage = gimage;
  p.g = make_geom(H, W);
  p.B = B;
  p.tiles_x = (W + kTW - 1) / kTW;
  p.tiles_y = (H + kTH - 1) / kTH;
  const long tiles = (long)B * p.tiles_x * p.tiles_y;
  FD_REQUIRE(tiles < (1L << 31), "warp_win_bwd: too many tiles");
  p.ntiles = (int)tiles;
  static const int dbg = fd_diag_bits("FD_WARP_WIN_DBG");
  p.dbg = dbg;
  CUtensorMap map_in, map_grad;
  const uint64_t dims[3] = {(uint64_t)W, (uint64_t)H, (uint64_t)B * kC};
  const uint64_t str[2] = {(uint64_t)W * 4, (uint64_t)H * W * 4};
  const uint32_t box[3] = {(uint32_t)kWW, (uint32_t)kWH, 1u};
  if (int e = make_tmap_f32_plain(&map_in, frame2, 3, dims, str, box)) return e;
  if (int e = make_tmap_f32_plain(&map_grad, gimage != nullptr ? (const void*)gimage : (const void*)frame2, 3, dims, str, box, kDiag && (p.dbg & 32) != 0)) return e;
  const int grid = (int)(tiles < FD_NUM_SMS ? tiles : FD_NUM_SMS);
  static bool attr_done[2] = {false, false};
  if (mode == 0) {
    if (!attr_done[0]) {
      FD_CUDA(cudaFuncSetAttribute(warp_win_bwd_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
      attr_done[0] = true;
    }
    warp_win_bwd_kernel<0><<<grid, kThreads, kSmemBytes, st>>>(map_in, map_grad, p);
  } else {
    if (!attr_done[1]) {
      FD_CUDA(cudaFuncSetAttribute(warp_win_bwd_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
      attr_done[1] = true;
    }
    warp_win_bwd_kernel<1><<<grid, kThreads, kSmemBytes, st>>>(map_in, map_grad, p);
  }
  FD_LAUNCH_CHECK();
  return FD_OK;
}
