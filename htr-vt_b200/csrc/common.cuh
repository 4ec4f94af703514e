// Shared device helpers for the HTR-VT sm_100a kernels: error codes, warp reductions,
// mbarrier / TMA / tcgen05 inline-PTX wrappers.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#define HTRVT_OK 0
#define HTRVT_ERR_SHAPE (-1)
#define HTRVT_ERR_ALIGN (-2)
#define HTRVT_ERR_ARCH (-3)
#define HTRVT_ERR_LAUNCH (-4)
#define HTRVT_ERR_WORKSPACE (-5)
#define HTRVT_ERR_DRIVER (-6)

// every kernel launch of the library is followed by HTRVT_LAUNCH_CHECK(): it counts the launch
// (htrvt_launch_count(), used by bench.py's gpu_launches) and converts launch errors to a status.
extern "C" unsigned long long htrvt_launch_counter;
#define HTRVT_LAUNCH_CHECK()                                   \
  do {                                                         \
    ++htrvt_launch_counter;                                    \
    cudaError_t e__ = cudaGetLastError();                      \
    if (e__ != cudaSuccess) return HTRVT_ERR_LAUNCH;           \
  } while (0)


// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute: remember what was set per (call site, device)
// so that one process driving several GPUs configures the kernel on each of them.  Evaluates to true on success.
#define HTRVT_ENSURE_SMEM(kern, bytes)                                                                       \
  ([&]() -> bool {                                                                                           \
    static int done__[64] = {0};                                                                             \
    int dev__ = 0;                                                                                           \
    cudaGetDevice(&dev__);                                                                                   \
    dev__ &= 63;                                                                                             \
    const int want__ = static_cast<int>(bytes);                                                              \
    if (done__[dev__] >= want__ && done__[dev__] > 0) return true;                                           \
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, want__) != cudaSuccess)      \
      return false;                                                                                          \
    done__[dev__] = want__;                                                                                  \
    return true;                                                                                             \
  }())

namespace htrvt {

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Block-wide sum for blockDim.x a multiple of 32 (<= 1024).  `red` is >= 33 floats of smem.
__device__ __forceinline__ float block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();                      // protect `red` from a previous call
  if (lane == 0) red[wid] = v;
  __syncthreads();
  if (wid == 0) {
    float t = lane < nw ? red[lane] : 0.f;
    t = warp_sum(t);
    if (lane == 0) red[32] = t;
  }
  __syncthreads();
  return red[32];
}

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2f(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack_bf16(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}

// IEEE fp16 pairs: the storage format of the FORWARD stem tensors (activations, raw conv outputs, forward weight
// copies).  Same 16 bits and the same tensor-core rate as bf16 with 3 more mantissa bits; these quantities are
// bounded (BatchNorm keeps them O(1)), gradients stay bf16 for their range.  Conversions saturate at +-65504.
__device__ __forceinline__ uint32_t pack_f16(float a, float b) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));   // first source -> upper half
  return r;
}
__device__ __forceinline__ float2 unpack_f16(uint32_t u) {
  return __half22float2(*reinterpret_cast<__half2*>(&u));
}
__device__ __forceinline__ float f16_bits_to_float(uint16_t h) { return __half2float(__ushort_as_half(h)); }

// ---------------------------------------------------------------------------------------------
// GELU (erf form, nn.GELU default used by timm Mlp) - shared by the fused GEMM epilogues and the stand-alone kernels
// ---------------------------------------------------------------------------------------------
// Phi(u) (standard normal CDF, i.e. the erf form of nn.GELU) and e = exp(-u^2/2) with two MUFU ops and six FMAs:
// erf(z) = 1 - (a1 t + ... + a5 t^5) exp(-z^2), t = 1/(1 + p z)  (Abramowitz-Stegun 7.1.26, |err| <= 1.5e-7 - far
// below the bf16 output resolution).  libm's erff costs ~2x the instructions, which made these two streaming kernels
// instruction bound (~3.3 TB/s); the exponential is shared with the density term of the backward.
__device__ __forceinline__ void gelu_parts(float u, float& cdf, float& e) {
  const float z = fabsf(u) * 0.70710678118654752f;
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.0f)));
  e = ex2f(u * u * -0.72134752044448170f);          // exp(-u^2 / 2)
  float p = fmaf(t, 1.061405429f, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  const float h = 0.5f * p * t * e;                 // 1 - Phi(|u|)
  cdf = u >= 0.f ? 1.0f - h : h;
}
__device__ __forceinline__ float gelu_val(float u) {
  float c, e;
  gelu_parts(u, c, e);
  return u * c;
}
__device__ __forceinline__ float gelu_grad(float u) {
  float c, e;
  gelu_parts(u, c, e);
  return fmaf(u * 0.3989422804014327f, e, c);
}
// gelu(u) and gelu'(u) from one evaluation of (Phi, exp): the training forward stores both
__device__ __forceinline__ void gelu_val_grad(float u, float& val, float& grad) {
  float c, e;
  gelu_parts(u, c, e);
  val = u * c;
  grad = fmaf(u * 0.3989422804014327f, e, c);
}

// ---------------------------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ---------------------------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor), tile mode, completion on an mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const void* desc) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(desc)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const void* desc, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const void* desc, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const void* desc, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* dst, const void* desc, uint64_t* bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3), "r"(c4)
      : "memory");
}

// multicast variant: the box lands at the same CTA-relative offset in every CTA of `mask`, and each destination
// CTA's mbarrier (same offset) receives the complete_tx
__device__ __forceinline__ void tma_load_5d_mc(void* dst, const void* desc, uint64_t* bar, int c0, int c1, int c2,
                                               int c3, int c4, uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2], %8;"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3), "r"(c4), "h"(mask)
      : "memory");
}

// CTA-pair (cta_group::2) variant: the box lands in the EXECUTING CTA's smem, the complete_tx goes to the mbarrier
// of the pair's leader (even CTA): clearing bit 24 of a shared::cluster address selects the even CTA's copy.
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ void tma_load_5d_pair(void* dst, const void* desc, uint64_t* bar, int c0, int c1, int c2,
                                                 int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0),
      "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
// arrive on the leader CTA's copy of `bar` (from either CTA of the pair)
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}

// ---------------------------------------------------------------------------------------------
// thread-block clusters
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {       // every thread of every CTA of the cluster
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {   // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {     // same warp as alloc
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc];  kind::f16 covers bf16 inputs with fp32 accumulation.
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// ... and on the same-offset mbarrier of every CTA in `mask` (smem slots shared through TMA multicast)
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"(mask)
      : "memory");
}
// ---- cta_group::2: one MMA spans the CTA pair (M = 256: 128 rows per CTA, each CTA holds half of B) ----------
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {   // same warp id in both CTAs
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of the pair's MMAs, signalled on the same-offset mbarrier of every CTA in `mask`
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"(mask)
      : "memory");
}
// TMEM -> registers: each thread reads its own lane (row), 16 consecutive 32-bit columns.
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor for tcgen05.mma (SWIZZLE_128B, version 1).
//  K-major tile  (rows x 64 bf16, one 128-byte row per MN index, 8-row groups of 1024 B):
//      SBO = 1024 B (next 8-row group), LBO unused.
//  MN-major tile (64 MN elements = 128 B contiguous per K index, 8 K-rows per 1024-B atom):
//      SBO = 1024 B (next 8 K indices), LBO = byte distance between 64-wide MN atoms.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= 1ull << 46;                       // descriptor version (Blackwell)
  d |= 2ull << 61;                       // SWIZZLE_128B
  return d;
}
// A K-major SWIZZLE_128B operand may start at ANY 128-byte row of a tile that TMA staged at a 1024-byte boundary
// (a shifted window of a larger tile): just move the start address.  tcgen05 applies the 128B XOR to the absolute
// shared-memory address bits, exactly as TMA did when writing, so the descriptor's base-offset field stays 0
// (setting it to (addr >> 7) & 7 double-shifts the pattern: measured, gemm.cu window reuse).
// MN-major tile under SWIZZLE_64B: 32 MN elements = 64 B contiguous per K index, 8 K-rows per 512-B atom:
//      SBO = 512 B (next 8 K indices), LBO = byte distance between 32-wide MN atoms.
__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= 1ull << 46;
  d |= 4ull << 61;                       // SWIZZLE_64B
  return d;
}
// Instruction descriptor: bf16 x bf16 -> fp32, M x N tile, operand major-ness (0 = K, 1 = MN).
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn, int b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a_mn) << 15) |
         (static_cast<uint32_t>(b_mn) << 16) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}

// Argument rules of the windowed variant's attention (attention2.cu), shared by its 16-bit entry and the fp32 one
// (exact.cu) so both precisions accept the same models and lines: head_dim 128, 1 <= T <= 256, window 0 or 16, shift 0
// for global blocks and a multiple of 8 below the window otherwise, a bias table of 2 * Prel - 1 <= 511 rows with
// Prel >= T.  HTRVT_OK or HTRVT_ERR_SHAPE.
int attention2_check(int B, int H, int T, int hd, int window, int shift, int Prel, const void* table);

}  // namespace htrvt
