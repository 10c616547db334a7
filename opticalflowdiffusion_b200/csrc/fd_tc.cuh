// sm_100a building blocks shared by the tensor-core kernels: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (alloc / mma / commit / ld) wrappers as inline PTX, UMMA descriptors, and the host-side
// tensor-map encoder (driver entry point fetched through the runtime, no link-time libcuda).
#pragma once

#include <cuda.h>

#include "fd_common.cuh"

namespace fdtc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// One elected lane of a fully converged warp (elect.sync).  The single-thread issue sites (TMA, tcgen05.mma / .commit) use
// this instead of `lane == 0`: under `if (lane == 0)` the compiler cannot prove that the uniform-datapath operands of
// UTCHMMA / UTCBAR / UTMALDG are warp-uniform and wraps EVERY such instruction in an ELECT + BRA.U.ANY waterfall loop
// (measured with ncu's source view on the N = 128 tiles: ~600 cycles to issue the 4 MMAs + 2 commits of a K-block that
// occupy the tensor pipe for 256); with elect.sync the issue sequence is straight-line SASS.
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

// Identity the compiler cannot see through: keeps a value in a general register (and out of the uniform datapath) until
// the instruction that consumes it.
__device__ __forceinline__ int opaque32(int x) {
  int y;
  asm volatile("mov.b32 %0, %1;" : "=r"(y) : "r"(x));
  return y;
}
__device__ __forceinline__ uint64_t opaque64(uint64_t x) {
  uint64_t y;
  asm volatile("mov.b64 %0, %1;" : "=l"(y) : "l"(x));
  return y;
}

// ---- mbarrier ----------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (and surfaces as a CUDA error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {
      printf("libflowdiff: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", blockIdx.x, threadIdx.x,
             bar, parity);
      __trap();
    }
  }
}

// ---- TMA -----------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(m), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
      "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst),
      "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(dst),
      "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

// smem -> global tensor store (clips to the tensor bounds); bulk-group completion
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3, int c4) {
  asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];" ::"l"(m), "r"(src),
               "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// make generic-proxy shared-memory writes visible to the async proxy (TMA) before it reads them
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- tcgen05 ---------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate, issued by ONE thread
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the mbarrier once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp receives lane (row) i
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major operand tile, rows of 64 bf16 (128 B) written by TMA with 128-byte swizzle:
// 8-row groups are 1024 B apart (SBO), LBO unused, descriptor version 1 (sm_100), layout SWIZZLE_128B.
// MEASURED on B200 (the strip conv's shifted-start descriptors): the tensor core applies the 128B swizzle
// XOR to the ABSOLUTE shared-memory address bits [7:9], exactly like TMA does when writing, so a descriptor may
// start at any 128-byte row of a 1024-byte-aligned TMA tile (rows shifted by 1 or 2 pixels for the conv taps)
// with base_offset = 0; setting base_offset = (addr >> 7) & 7 for such starts gives WRONG results.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(1024u >> 4) << 32;
  d |= 1ull << 46;
  d |= 2ull << 61;
  return d;
}
// instruction descriptor: D fp32, A/B bf16, both K-major, M x N
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- host: tensor maps -----------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = (EncodeTiledFn)p;
  }
  return fn;
}

// bf16 tensor, up to 5 dims (dim 0 innermost / contiguous), 128B swizzle, zero fill out of bounds.
// strides_bytes[i] is the byte stride of dim i+1.
inline int make_tmap_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                          const uint64_t* strides_bytes, const uint32_t* box) {
  EncodeTiledFn fn = get_encode_tiled();
  if (!fn) {
    fd_set_error("cuTensorMapEncodeTiled is unavailable (driver entry point lookup failed)");
    return FD_ECUDA;
  }
  cuuint64_t gd[5];
  cuuint64_t gs[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gd[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
  }
  for (int i = 0; i + 1 < rank; ++i) gs[i] = strides_bytes[i];
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    fd_set_error("cuTensorMapEncodeTiled failed (%d): rank %d dims [%llu %llu %llu %llu %llu] box [%u %u %u %u %u]",
                 (int)r, rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
                 (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0),
                 (unsigned long long)(rank > 4 ? dims[4] : 0), box[0], rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0,
                 rank > 3 ? box[3] : 0, rank > 4 ? box[4] : 0);
    return FD_ECUDA;
  }
  return FD_OK;
}

// fp32 tensor, up to 5 dims, NO swizzle (plain row-major box in shared memory), zero fill out of bounds (negative start
// coordinates included): the sampled-frame windows of fd_warp_win.cu.
inline int make_tmap_f32_plain(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                               const uint32_t* box, bool l2_promotion = true) {
  EncodeTiledFn fn = get_encode_tiled();
  if (!fn) {
    fd_set_error("cuTensorMapEncodeTiled is unavailable (driver entry point lookup failed)");
    return FD_ECUDA;
  }
  cuuint64_t gd[5];
  cuuint64_t gs[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gd[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
  }
  for (int i = 0; i + 1 < rank; ++i) gs[i] = strides_bytes[i];
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                  l2_promotion ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B : CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    fd_set_error("cuTensorMapEncodeTiled (fp32) failed (%d): rank %d dims [%llu %llu %llu] box [%u %u %u]", (int)r, rank,
                 (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
                 (unsigned long long)(rank > 2 ? dims[2] : 0), box[0], rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0);
    return FD_ECUDA;
  }
  return FD_OK;
}

}  // namespace fdtc
