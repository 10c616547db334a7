// Backward bilinear warp (warp.py:95-119 of the reference) and the fused
// warp + Charbonnier photometric + end-point-error objective (losses.py:3-6,46-47).
//
// Gather/scatter work on fp32 NCHW planes.  The FORWARD operations on three-channel frames with W % 4 == 0 run the
// shared-memory window kernels of fd_warp_win.cu (TMA-staged frame, 1.5-2x faster on the config-#4 white-noise flow);
// the kernels in this file serve every other shape and all the backward passes.  Layout choices:
//   * one thread owns VEC (2 when W is even, else 1) consecutive pixels of a row, so flow / flow_gt /
//     frame1 / out / mask move as wide coalesced accesses; a block walks (row, segment) jobs, no per-thread divisions;
//   * the 4-tap gathers of the warped frame go through the read-only path (L1/L2 resident: a
//     warp's taps fall in a few rows of the source plane);
//   * the scatter of the image gradient merges contributions that hit the same address inside a
//     thread and across neighbouring lanes (shuffle) before falling back to red.global.add.f32.
//
// The coordinate / weight / accumulation sequence is written with explicit round-to-nearest
// intrinsics in the exact order ATen's CPU grid_sampler_2d evaluates it, which makes the forward
// bit-identical to the reference's CPU output (oracle/flowdiff_oracle.py:backwarp).
#include <initializer_list>

#include "fd_warp_common.cuh"

using namespace fdwarp;

namespace {

template <int VEC>
struct Vec;
template <>
struct Vec<1> {
  float v[1];
  __device__ __forceinline__ void load(const float* p) { v[0] = __ldg(p); }
  __device__ __forceinline__ void store(float* p) const { *p = v[0]; }
};
template <>
struct Vec<2> {
  float v[2];
  __device__ __forceinline__ void load(const float* p) {
    const float2 t = __ldg(reinterpret_cast<const float2*>(p));
    v[0] = t.x; v[1] = t.y;
  }
  __device__ __forceinline__ void store(float* p) const { *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]); }
};

// Work decomposition without per-thread divisions.  A "row job" = (image row r = b * H + y, segment of blockDim.x * VEC
// pixels of it); blocks walk the jobs grid-stride, thread t of a block owns VEC consecutive pixels of the segment.  The first
// version mapped a flat 64-bit item index to (b, y, x) with three 64-bit divisions PER THREAD per item: ncu showed 298
// executed instructions per pixel in the fused photometric forward, most of them division emulation (IMAD chains + CALLs).
// Here the two divisions are 32-bit, once per job, on block-uniform values; offsets inside a plane are 32-bit (H * W < 2^31
// is checked on the host), only the plane base is 64-bit.
struct RowJob {
  int b, y, x;      // x = first of the thread's VEC pixels
  bool valid;       // x < W (ragged last segment)
};
template <int VEC>
__device__ __forceinline__ RowJob row_job(unsigned job, unsigned segs, unsigned H, int W) {
  const unsigned row = job / segs, seg = job - row * segs;
  const unsigned b = row / H;
  RowJob r;
  r.b = (int)b;
  r.y = (int)(row - b * H);
  r.x = (int)((seg * blockDim.x + threadIdx.x) * VEC);
  r.valid = r.x < W;
  return r;
}
static unsigned row_segs(int W, int vec, int threads) { return (unsigned)((W / vec + threads - 1) / threads); }

// ---------------------------------------------------------------------------------------------
// forward: out, mask
// ---------------------------------------------------------------------------------------------
template <int VEC, int CT>
__global__ void __launch_bounds__(256, 4) backwarp_fwd_kernel(const float* __restrict__ image,
                                                           const float* __restrict__ flow,
                                                           float* __restrict__ out, float* __restrict__ mask,
                                                           int B, int C, BwGeom g, unsigned segs, unsigned jobs) {
  const int H = g.H, W = g.W;
  const long HW = (long)H * W;
  const BwDiv dv = bw_divisors(g);
  for (unsigned job = blockIdx.x; job < jobs; job += gridDim.x) {
    const RowJob rj = row_job<VEC>(job, segs, (unsigned)H, W);
    if (!rj.valid) continue;
    const int b = rj.b, y = rj.y, x = rj.x;
    const int pix = y * W + x;
    Vec<VEC> fdy, fdx;
    fdy.load(flow + ((long)b * 2 + 0) * HW + pix);
    fdx.load(flow + ((long)b * 2 + 1) * HW + pix);
    BwTaps t[VEC];
    Vec<VEC> m;
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      bw_taps(fdx.v[j], fdy.v[j], x + j, y, g, dv, t[j]);
      m.v[j] = bw_mask(t[j]);
    }
    const int Cn = CT > 0 ? CT : C;          // CT = 3: the RGB case unrolled, all three channels' gathers in flight at once
#pragma unroll
    for (int c = 0; c < Cn; ++c) {
      const float* plane = image + ((long)b * C + c) * HW;
      Vec<VEC> o;
#pragma unroll
      for (int j = 0; j < VEC; ++j) o.v[j] = bw_sample(bw_gather(plane, t[j], W), t[j]);
      o.store(out + ((long)b * C + c) * HW + pix);
      if (mask != nullptr) m.store(mask + ((long)b * C + c) * HW + pix);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// backward of sum(out * gout): gimage (scatter), gflow (gather)
// ---------------------------------------------------------------------------------------------
template <int VEC, int CT>
__global__ void __launch_bounds__(256, 3) backwarp_bwd_kernel(const float* __restrict__ image,
                                                           const float* __restrict__ flow,
                                                           const float* __restrict__ gout,
                                                           float* __restrict__ gimage, float* __restrict__ gflow,
                                                           int B, int C, BwGeom g, unsigned segs, unsigned jobs) {
  const int H = g.H, W = g.W;
  const long HW = (long)H * W;
  const BwDiv dv = bw_divisors(g);
  for (unsigned job = blockIdx.x; job < jobs; job += gridDim.x) {        // (whole warps stay together: fd_scatter_merged)
    const RowJob rj = row_job<VEC>(job, segs, (unsigned)H, W);
    const bool valid = rj.valid;
    const int b = rj.b, y = rj.y, x = valid ? rj.x : 0;
    const int pix = y * W + x;
    Vec<VEC> fdy, fdx;
#pragma unroll
    for (int j = 0; j < VEC; ++j) fdy.v[j] = fdx.v[j] = 0.f;
    if (valid) {
      fdy.load(flow + ((long)b * 2 + 0) * HW + pix);
      fdx.load(flow + ((long)b * 2 + 1) * HW + pix);
    }
    BwTaps t[VEC];
    float dix[VEC], diy[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      bw_taps(fdx.v[j], fdy.v[j], x + j, y, g, dv, t[j]);
      dix[j] = diy[j] = 0.f;
    }
    const int Cn = CT > 0 ? CT : C;
#pragma unroll
    for (int c = 0; c < Cn; ++c) {
      const long plane_off = ((long)b * C + c) * HW;
      Vec<VEC> go;
#pragma unroll
      for (int j = 0; j < VEC; ++j) go.v[j] = 0.f;
      if (valid) go.load(gout + plane_off + pix);
      if (gflow != nullptr && valid) {
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          const BwVals v = bw_gather(image + plane_off, t[j], W);
          dix[j] += go.v[j] * ((v.ne - v.nw) * t[j].sy + (v.se - v.sw) * t[j].ny);
          diy[j] += go.v[j] * ((v.sw - v.nw) * t[j].ex + (v.se - v.ne) * t[j].wx);
        }
      }
      if (gimage != nullptr) {
        int a0[2 * VEC], a1[2 * VEC];
        float v0[2 * VEC], v1[2 * VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          const int r0 = t[j].y0 * W + t[j].x0;
          a0[2 * j] = (valid && t[j].okx0 && t[j].oky0) ? r0 : -1;
          a0[2 * j + 1] = (valid && t[j].okx1 && t[j].oky0) ? r0 + 1 : -1;
          a1[2 * j] = (valid && t[j].okx0 && t[j].oky1) ? r0 + W : -1;
          a1[2 * j + 1] = (valid && t[j].okx1 && t[j].oky1) ? r0 + W + 1 : -1;
          v0[2 * j] = go.v[j] * t[j].nw;
          v0[2 * j + 1] = go.v[j] * t[j].ne;
          v1[2 * j] = go.v[j] * t[j].sw;
          v1[2 * j + 1] = go.v[j] * t[j].se;
        }
        fd_scatter_merged<2 * VEC>(gimage + plane_off, a0, v0);
        fd_scatter_merged<2 * VEC>(gimage + plane_off, a1, v1);
      }
    }
    if (gflow != nullptr && valid) {
      Vec<VEC> gy, gx;
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        gx.v[j] = ((dix[j] * g.half_w) / g.wm1n) * 2.f;
        gy.v[j] = ((diy[j] * g.half_h) / g.hm1n) * 2.f;
      }
      gy.store(gflow + ((long)b * 2 + 0) * HW + pix);
      gx.store(gflow + ((long)b * 2 + 1) * HW + pix);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// fused warp + photometric + EPE
// ---------------------------------------------------------------------------------------------
constexpr int kPhotoThreads = 256;

static int photo_grid(long items) {        // items = row jobs
  long blocks = items;
  const long cap = (long)FD_NUM_SMS * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

template <int VEC, int CT>
__global__ void __launch_bounds__(kPhotoThreads, 4) photo_epe_fwd_kernel(
    const float* __restrict__ frame1, const float* __restrict__ frame2, const float* __restrict__ flow,
    const float* __restrict__ flow_gt, float* __restrict__ partials, int B, int C, BwGeom g, unsigned segs, unsigned jobs) {
  __shared__ float red[3 * 32];
  const int H = g.H, W = g.W;
  const long HW = (long)H * W;
  const BwDiv dv = bw_divisors(g);
  float s[3] = {0.f, 0.f, 0.f};
  for (unsigned job = blockIdx.x; job < jobs; job += gridDim.x) {
    const RowJob rj = row_job<VEC>(job, segs, (unsigned)H, W);
    if (!rj.valid) continue;
    const int b = rj.b, y = rj.y, x = rj.x;
    const int pix = y * W + x;
    const long fo = (long)b * 2 * HW + pix;
    Vec<VEC> f0, f1, g0, g1;
    f0.load(flow + fo);
    f1.load(flow + fo + HW);
    g0.load(flow_gt + fo);
    g1.load(flow_gt + fo + HW);
    BwTaps t[VEC];
    float m[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      bw_taps(f1.v[j], f0.v[j], x + j, y, g, dv, t[j]);
      m[j] = bw_mask(t[j]);
      const float du = f0.v[j] - g0.v[j], dv = f1.v[j] - g1.v[j];
      const float e2 = du * du + dv * dv;
      s[2] += e2 > 0.f ? e2 * rsqrtf(e2) : 0.f;
    }
    const int Cn = CT > 0 ? CT : C;
#pragma unroll
    for (int c = 0; c < Cn; ++c) {
      const long po = ((long)b * C + c) * HW;
      Vec<VEC> a;
      a.load(frame1 + po + pix);
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const float wv = bw_sample(bw_gather(frame2 + po, t[j], W), t[j]);
        const float d = a.v[j] - wv;
        const float q = d * d + 1e-6f;
        s[0] += m[j] * (q * rsqrtf(q));          // sqrt(q), q >= 1e-6: 2-ulp approximation, one MUFU instead of IEEE sqrt
        s[1] += m[j];
      }
    }
  }
  fd_block_sum<3>(s, red);
  if (threadIdx.x == 0) {
    partials[blockIdx.x * 3 + 0] = s[0];
    partials[blockIdx.x * 3 + 1] = s[1];
    partials[blockIdx.x * 3 + 2] = s[2];
  }
}

// fixed-order (deterministic) final reduction of per-block partials, in double
template <int NV>
__global__ void __launch_bounds__(256) finalize_sums_kernel(const float* __restrict__ partials, int nblocks,
                                                            float* __restrict__ sums, float extra, int extra_slot) {
  __shared__ double sh[NV][256];
  double acc[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) acc[i] = 0.0;
  for (int k = threadIdx.x; k < nblocks; k += 256)
#pragma unroll
    for (int i = 0; i < NV; ++i) acc[i] += (double)partials[k * NV + i];
#pragma unroll
  for (int i = 0; i < NV; ++i) sh[i][threadIdx.x] = acc[i];
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o)
#pragma unroll
      for (int i = 0; i < NV; ++i) sh[i][threadIdx.x] += sh[i][threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) sums[i] = (float)sh[i][0];
    if (extra_slot >= 0) sums[extra_slot] = extra;
  }
}

template <int VEC, int CT>
__global__ void __launch_bounds__(256, 3) photo_epe_bwd_kernel(
    const float* __restrict__ frame1, const float* __restrict__ frame2, const float* __restrict__ flow,
    const float* __restrict__ flow_gt, const float* __restrict__ sums, float g_photo, float g_epe,
    float* __restrict__ gflow, float* __restrict__ gframe2, int B, int C, BwGeom g, unsigned segs, unsigned jobs) {
  const int H = g.H, W = g.W;
  const long HW = (long)H * W;
  const BwDiv dv = bw_divisors(g);
  const float kp = g_photo / __ldg(sums + 1);
  const float ke = g_epe / __ldg(sums + 3);
  for (unsigned job = blockIdx.x; job < jobs; job += gridDim.x) {        // (whole warps stay together: fd_scatter_merged)
    const RowJob rj = row_job<VEC>(job, segs, (unsigned)H, W);
    const bool valid = rj.valid;
    const int b = rj.b, y = rj.y, x = valid ? rj.x : 0;
    const int pix = y * W + x;
    const long fo = (long)b * 2 * HW + pix;
    Vec<VEC> f0, f1, g0, g1;
#pragma unroll
    for (int j = 0; j < VEC; ++j) f0.v[j] = f1.v[j] = g0.v[j] = g1.v[j] = 0.f;
    if (valid) {
      f0.load(flow + fo);
      f1.load(flow + fo + HW);
      g0.load(flow_gt + fo);
      g1.load(flow_gt + fo + HW);
    }
    BwTaps t[VEC];
    float m[VEC], dix[VEC], diy[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      bw_taps(f1.v[j], f0.v[j], x + j, y, g, dv, t[j]);
      m[j] = bw_mask(t[j]);
      dix[j] = diy[j] = 0.f;
    }
    const int Cn = CT > 0 ? CT : C;
#pragma unroll
    for (int c = 0; c < Cn; ++c) {
      const long po = ((long)b * C + c) * HW;
      Vec<VEC> a;
#pragma unroll
      for (int j = 0; j < VEC; ++j) a.v[j] = 0.f;
      if (valid) a.load(frame1 + po + pix);
      float gw[VEC];
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        gw[j] = 0.f;
        if (valid) {
          const BwVals v = bw_gather(frame2 + po, t[j], W);
          const float d = a.v[j] - bw_sample(v, t[j]);
          gw[j] = -kp * m[j] * d / sqrtf(d * d + 1e-6f);   // dL/dwarped
          dix[j] += gw[j] * ((v.ne - v.nw) * t[j].sy + (v.se - v.sw) * t[j].ny);
          diy[j] += gw[j] * ((v.sw - v.nw) * t[j].ex + (v.se - v.ne) * t[j].wx);
        }
      }
      if (gframe2 != nullptr) {
        int a0[2 * VEC], a1[2 * VEC];
        float v0[2 * VEC], v1[2 * VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          const int r0 = t[j].y0 * W + t[j].x0;
          const bool on = valid && gw[j] != 0.f;
          a0[2 * j] = (on && t[j].okx0 && t[j].oky0) ? r0 : -1;
          a0[2 * j + 1] = (on && t[j].okx1 && t[j].oky0) ? r0 + 1 : -1;
          a1[2 * j] = (on && t[j].okx0 && t[j].oky1) ? r0 + W : -1;
          a1[2 * j + 1] = (on && t[j].okx1 && t[j].oky1) ? r0 + W + 1 : -1;
          v0[2 * j] = gw[j] * t[j].nw;
          v0[2 * j + 1] = gw[j] * t[j].ne;
          v1[2 * j] = gw[j] * t[j].sw;
          v1[2 * j + 1] = gw[j] * t[j].se;
        }
        fd_scatter_merged<2 * VEC>(gframe2 + po, a0, v0);
        fd_scatter_merged<2 * VEC>(gframe2 + po, a1, v1);
      }
    }
    if (gflow != nullptr && valid) {
      Vec<VEC> gy, gx;
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const float du = f0.v[j] - g0.v[j], dv = f1.v[j] - g1.v[j];
        const float nrm = sqrtf(du * du + dv * dv);
        const float inv = nrm > 0.f ? ke / nrm : 0.f;
        gy.v[j] = ((diy[j] * g.half_h) / g.hm1n) * 2.f + du * inv;
        gx.v[j] = ((dix[j] * g.half_w) / g.wm1n) * 2.f + dv * inv;
      }
      gy.store(gflow + fo);
      gx.store(gflow + fo + HW);
    }
  }
}

static int stream_grid(long items, int threads) {        // items = row jobs (one block-iteration each)
  (void)threads;
  long blocks = items;
  const long cap = (long)FD_NUM_SMS * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

// pixels per thread: 2 consecutive pixels when W allows
static int pick_vec(int W) { return W % 2 == 0 ? 2 : 1; }

// kernel<VEC, CT> for the runtime (vec, C): CT = 3 unrolls the RGB case
#define FD_WARP_DISPATCH(kern, ...)                       \
  do {                                                    \
    if (vec == 2) {                                       \
      if (C == 3) kern<2, 3> __VA_ARGS__; else kern<2, 0> __VA_ARGS__; \
    } else {                                              \
      if (C == 3) kern<1, 3> __VA_ARGS__; else kern<1, 0> __VA_ARGS__; \
    }                                                     \
  } while (0)

// Exhaustive check of bw_div_rn (fd_warp_common.cuh) against __fdiv_rn: all 2^32 numerator bit patterns for one divisor.
__global__ void __launch_bounds__(256) div_selftest_kernel(float c, unsigned long long* __restrict__ mismatches) {
  const BwRcp rc = bw_rcp(c);
  unsigned long long bad = 0;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < (1ull << 32);
       i += (unsigned long long)gridDim.x * blockDim.x) {
    const float a = __uint_as_float((unsigned)i);
    const unsigned got = __float_as_uint(bw_div_rn(a, rc)), want = __float_as_uint(__fdiv_rn(a, c));
    const bool both_nan = (got & 0x7fffffffu) > 0x7f800000u && (want & 0x7fffffffu) > 0x7f800000u;
    if (got != want && !both_nan) ++bad;
  }
  bad = __reduce_add_sync(0xffffffffu, (unsigned)bad);      // (per-thread counts stay far below 2^32 / 32)
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(mismatches, bad);
}

// pick_vec restricted by the alignment of the tensors (a view at an odd float offset is a legal argument): VEC consecutive
// floats are moved as one access, so every plane base must be a multiple of 4 * VEC bytes (H * W * 4 is, when VEC | W)
static int vec_for(int W, std::initializer_list<const void*> ptrs) {
  int v = pick_vec(W);
  for (const void* q : ptrs)
    while (v > 1 && q != nullptr && (reinterpret_cast<uintptr_t>(q) % (4u * (unsigned)v)) != 0) v >>= 1;
  return v;
}

static int check_dims(int B, int C, int H, int W) {
  FD_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "backwarp: non-positive dimension B=%d C=%d H=%d W=%d", B, C, H, W);
  FD_REQUIRE((long)H * W < (1L << 31), "backwarp: plane too large");
  return FD_OK;
}

}  // namespace

// fd_warp_win.cu: forward kernels with the sampled frame staged in shared memory by TMA (three-channel frames, W % 4 == 0)
int fd_warp_win_grid(int B, int H, int W);
int fd_warp_fwd_win(int mode, const float* frame1, const float* frame2, const float* flow, const float* flow_gt, float* out,
                    float* mask, float* partials, float* sums, int B, int H, int W, cudaStream_t st);

int fd_warp_bwd_win(int mode, const float* frame1, const float* frame2, const float* flow, const float* flow_gt, const float* gout,
                    const float* sums, float g_photo, float g_epe, float* gflow, float* gimage, int B, int H, int W, cudaStream_t st);

int fd_warp_bwd_win2(int mode, const float* frame1, const float* frame2, const float* flow, const float* flow_gt, const float* gout,
                     const float* fsums, float g_photo, float g_epe, float* gflow, float* gimage, float* acc, int B, int H, int W,
                     cudaStream_t st);

// the window kernels take three-channel frames, W % 4 == 0 and 16-byte aligned planes; the gather kernels everything else
static bool use_win(int C, int W, const void* a, const void* b, const void* c, const void* d, const void* e2 = nullptr,
                    const void* f = nullptr) {
  auto al = [](const void* q) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  return C == 3 && W % 4 == 0 && W >= 64 && al(a) && al(b) && al(c) && al(d) && al(e2) && al(f);
}

extern "C" {

int fd_backwarp_fwd(const float* image, const float* flow, float* out, float* mask, int B, int C, int H, int W,
                    void* stream) {
  if (int e = check_dims(B, C, H, W)) return e;
  FD_REQUIRE(image && flow && out, "backwarp_fwd: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (use_win(C, W, image, flow, out, mask)) return fd_warp_fwd_win(0, nullptr, image, flow, nullptr, out, mask, nullptr, nullptr, B, H, W, st);
  const BwGeom g = make_geom(H, W);
  const int vec = vec_for(W, {image, flow, out, mask});
  const unsigned segs = row_segs(W, vec, 256);
  const long items = (long)B * H * segs;                       // row jobs
  FD_REQUIRE(items < (1L << 31), "backwarp: too many row segments");
  FD_WARP_DISPATCH(backwarp_fwd_kernel, <<<stream_grid(items, 256), 256, 0, st>>>(image, flow, out, mask, B, C, g, segs, (unsigned)items));
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_backwarp_bwd(const float* image, const float* flow, const float* gout, float* gimage, float* gflow, int B,
                    int C, int H, int W, void* stream) {
  if (int e = check_dims(B, C, H, W)) return e;
  FD_REQUIRE(image && flow && gout, "backwarp_bwd: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const BwGeom g = make_geom(H, W);
  if (gimage) FD_CUDA(cudaMemsetAsync(gimage, 0, sizeof(float) * (size_t)B * C * H * W, st));
  if (use_win(C, W, image, flow, gout, gimage, gflow))
    return fd_warp_bwd_win(0, nullptr, image, flow, nullptr, gout, nullptr, 0.f, 0.f, gflow, gimage, B, H, W, st);
  const int vec = vec_for(W, {image, flow, gout, gimage, gflow});
  const unsigned segs = row_segs(W, vec, 256);
  const long items = (long)B * H * segs;                       // row jobs
  FD_REQUIRE(items < (1L << 31), "backwarp: too many row segments");
  FD_WARP_DISPATCH(backwarp_bwd_kernel, <<<stream_grid(items, 256), 256, 0, st>>>(image, flow, gout, gimage, gflow, B, C, g, segs, (unsigned)items));
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_warp_div_selftest(float divisor, unsigned long long* mismatches, void* stream) {
  FD_REQUIRE(mismatches != nullptr, "warp_div_selftest: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  FD_CUDA(cudaMemsetAsync(mismatches, 0, sizeof(unsigned long long), st));
  div_selftest_kernel<<<FD_NUM_SMS * 8, 256, 0, st>>>(divisor, mismatches);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

// Backward passes with a caller-provided workspace of fd_warp_bwd_workspace_floats(B, H, W) floats (16-byte aligned): on
// three-channel frames with W % 4 == 0 the frame gradient is accumulated pixel-interleaved in it, one 128-bit reduction per
// tap (4 instead of 12 L2 reduction operations per pixel), and converted to the planar gradient by a second launch; every
// other shape runs the workspace-free entry points above.
size_t fd_warp_bwd_workspace_floats(int B, int H, int W) { return (size_t)4 * B * H * W; }

int fd_backwarp_bwd_ws(const float* image, const float* flow, const float* gout, float* gimage, float* gflow, float* workspace,
                       int B, int C, int H, int W, void* stream) {
  if (int e = check_dims(B, C, H, W)) return e;
  FD_REQUIRE(image && flow && gout, "backwarp_bwd_ws: null pointer");
  if (workspace != nullptr && use_win(C, W, image, flow, gout, gimage, gflow, workspace))
    return fd_warp_bwd_win2(2, nullptr, image, flow, nullptr, gout, nullptr, 0.f, 0.f, gflow, gimage, workspace, B, H, W,
                            (cudaStream_t)stream);
  return fd_backwarp_bwd(image, flow, gout, gimage, gflow, B, C, H, W, stream);
}

int fd_backwarp_photo_epe_bwd_ws(const float* frame1, const float* frame2, const float* flow, const float* flow_gt,
                                 const float* sums, float g_photo, float g_epe, float* gflow, float* gframe2, float* workspace,
                                 int B, int C, int H, int W, void* stream) {
  if (int e = check_dims(B, C, H, W)) return e;
  FD_REQUIRE(frame1 && frame2 && flow && flow_gt && sums, "photo_epe_bwd_ws: null pointer");
  if (workspace != nullptr && use_win(C, W, frame1, frame2, flow, flow_gt, gflow, gframe2) &&
      (reinterpret_cast<uintptr_t>(workspace) & 15) == 0)
    return fd_warp_bwd_win2(3, frame1, frame2, flow, flow_gt, nullptr, sums, g_photo, g_epe, gflow, gframe2, workspace, B, H, W,
                            (cudaStream_t)stream);
  return fd_backwarp_photo_epe_bwd(frame1, frame2, flow, flow_gt, sums, g_photo, g_epe, gflow, gframe2, B, C, H, W, stream);
}

size_t fd_photo_epe_workspace_floats(int B, int H, int W) {
  const long items = (long)B * H * row_segs(W, 1, 256);        // (the narrowest vector width: the largest grid)
  const size_t a = (size_t)photo_grid(items) * 3;
  const size_t c = (size_t)fd_warp_win_grid(B, H, W) * 3 + 4;      // + the 8-byte aligned 64-bit ticket word
  return a > c ? a : c;
}

int fd_backwarp_photo_epe_fwd(const float* frame1, const float* frame2, const float* flow, const float* flow_gt,
                              float* sums, float* partials, int B, int C, int H, int W, void* stream) {
  if (int e = check_dims(B, C, H, W)) return e;
  FD_REQUIRE(frame1 && frame2 && flow && flow_gt && sums && partials, "photo_epe_fwd: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (use_win(C, W, frame1, frame2, flow, flow_gt)) {
    return fd_warp_fwd_win(1, frame1, frame2, flow, flow_gt, nullptr, nullptr, partials, sums, B, H, W, st);
  }
  const BwGeom g = make_geom(H, W);
  const int vec = vec_for(W, {frame1, frame2, flow, flow_gt});
  const unsigned segs = row_segs(W, vec, 256);
  const long items = (long)B * H * segs;                       // row jobs
  FD_REQUIRE(items < (1L << 31), "backwarp: too many row segments");
  const int grid = photo_grid(items);
  FD_WARP_DISPATCH(photo_epe_fwd_kernel, <<<grid, kPhotoThreads, 0, st>>>(frame1, frame2, flow, flow_gt, partials, B, C, g, segs, (unsigned)items));
  FD_LAUNCH_CHECK();
  finalize_sums_kernel<3><<<1, 256, 0, st>>>(partials, grid, sums, (float)((double)B * H * W), 3);
  FD_LAUNCH_CHECK();
  return FD_OK;
}

int fd_backwarp_photo_epe_bwd(const float* frame1, const float* frame2, const float* flow, const float* flow_gt,
                              const float* sums, float g_photo, float g_epe, float* gflow, float* gframe2, int B,
                              int C, int H, int W, void* stream) {
  if (int e = check_dims(B, C, H, W)) return e;
  FD_REQUIRE(frame1 && frame2 && flow && flow_gt && sums, "photo_epe_bwd: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const BwGeom g = make_geom(H, W);
  if (gframe2) FD_CUDA(cudaMemsetAsync(gframe2, 0, sizeof(float) * (size_t)B * C * H * W, st));
  if (use_win(C, W, frame1, frame2, flow, flow_gt, gflow, gframe2))
    return fd_warp_bwd_win(1, frame1, frame2, flow, flow_gt, nullptr, sums, g_photo, g_epe, gflow, gframe2, B, H, W, st);
  const int vec = vec_for(W, {frame1, frame2, flow, flow_gt, gflow, gframe2});
  const unsigned segs = row_segs(W, vec, 256);
  const long items = (long)B * H * segs;                       // row jobs
  FD_REQUIRE(items < (1L << 31), "backwarp: too many row segments");
  FD_WARP_DISPATCH(photo_epe_bwd_kernel, <<<stream_grid(items, 256), 256, 0, st>>>(frame1, frame2, flow, flow_gt, sums, g_photo, g_epe, gflow, gframe2, B, C, g, segs, (unsigned)items));
  FD_LAUNCH_CHECK();
  return FD_OK;
}

}  // extern "C"
