// Attention of the windowed HTR-VT variant (model_window/model/HTR_VT.py:11-62, 114-154) for sm_100a:
// head_dim 128, sequence T <= 256, learned relative-position bias  table[(j - i) + P - 1][h]  added to the scaled
// scores, and two geometries:
//   * global   (window == 0): every query attends to all T keys (two 128-key blocks);
//   * windowed (window == 16): the sequence is rolled by -shift, cut into 16-token windows, attention runs inside
//     each window (bias indexed by the intra-window offset, the wrap-around window mixes head and tail tokens),
//     results roll back.  T need not be a multiple of 16: the reference zero-pads to Tp = ceil16(T), rolls tokens AND
//     the validity mask, masks the padded keys and strips the padded queries (:121-131, :49-56) - here padded tokens
//     are TMA out-of-bounds zeros, padded keys get -inf scores, padded query rows are never stored.
//     One CTA handles 128 consecutive ROLLED positions = 8 windows as ONE 128 x 128 tcgen05
//     score tile with a block-diagonal mask: the tensor core wastes 7/8 of a tile that is 0.03 % of the step, and
//     the kernel stays a single TMA -> tcgen05 -> TMEM pipeline instead of thousands of 16 x 16 problems.
// Attention dropout (attn_drop = 0.05 in train mode) is a counter-based hash of (seed, b, h, query token,
// key token), so the backward regenerates the mask instead of storing it.
//   fwd: CTA per (b, h, 128-query block); S = Q K^T (N = 128 or 256) in TMEM, softmax in registers, P (bf16) to the
//        K image's smem, O = P V.
//   bwd: CTA per (b, h, 128-key block) loops over the query blocks that see it: recompute S, dP = dO V^T,
//        dS = P o (dP - delta); dV += (P o M)^T dO and dK += dS^T Q accumulate in TMEM across query blocks,
//        dQ = dS K per pair (T > 128, global: bf16 partials per key block, summed by add_dq_kernel);
//        dTable[(j - i) + P - 1][h] += sum dS / scale.
#include "common.cuh"
#include <cuda.h>

namespace htrvt {

constexpr int kA2Threads = 160;            // warps 0-3: one thread per query/key row; warp 4: TMA + MMA issue
constexpr int kA2Hd = 128;
constexpr int kChunk128 = 128 * 128;       // bytes of a [128 rows][64 bf16] swizzled chunk image

struct Attn2P {
  int B, H, T;
  int Tp;                      // windowed: T padded to a multiple of the window (16); else T
  int nblk;                    // ceil(T / 128)
  int window, shift;           // window 0 (global) or 16
  int Prel;                    // relative-position table has 2 * Prel - 1 rows
  float scale;
  const float* table;          // [2*Prel-1][H] fp32 or null
  float* dtable;               // bwd: gradient of table (+=, atomics)
  __nv_bfloat16* out;          // fwd: [B, T, H*hd]
  float* lse;                  // [B, H, T]
  const __nv_bfloat16* o;      // bwd
  const __nv_bfloat16* dout;   // bwd
  __nv_bfloat16* dqkv;         // bwd: [B, T, 3, H, hd]
  __nv_bfloat16* dq_part;      // bwd, global T > 128: [nblk][B*T][H*hd] partial dQ per key block
  float drop_p;                // attention dropout probability (0 = off)
  unsigned long long seed;
};

__device__ __forceinline__ uint32_t hash_u32(uint32_t x) {          // murmur3 finaliser
  x ^= x >> 16; x *= 0x85ebca6bu; x ^= x >> 13; x *= 0xc2b2ae35u; x ^= x >> 16;
  return x;
}
// keep-scale of attention dropout for (b, h, query token, key token): 0 or 1 / (1 - p)
__device__ __forceinline__ float attn_keep(unsigned long long seed, int bh, int ti, int tj, float p, float inv_keep) {
  const uint32_t a = hash_u32(static_cast<uint32_t>(seed) ^ (static_cast<uint32_t>(bh) * 0x9e3779b9u));
  const uint32_t v = hash_u32(a ^ hash_u32(static_cast<uint32_t>(seed >> 32) + static_cast<uint32_t>(ti) * 65537u +
                                           static_cast<uint32_t>(tj)));
  return (static_cast<float>(v >> 8) * (1.0f / 16777216.0f)) < p ? 0.f : inv_keep;
}

__device__ __forceinline__ void store_row8(uint8_t* img, int chunk_bytes, int r, int c, int g, uint4 v) {
  *reinterpret_cast<uint4*>(img + c * chunk_bytes + r * 128 + ((g ^ (r & 7)) << 4)) = v;
}
__device__ __forceinline__ uint64_t d_kmajor(uint32_t img, int chunk_bytes, int k16) {     // MN = rows, K = cols
  return umma_desc_sw128(img + (k16 >> 2) * chunk_bytes + (k16 & 3) * 32, 16, 1024);
}
__device__ __forceinline__ uint64_t d_mnmajor(uint32_t img, int chunk_bytes, int k16) {    // MN = cols, K = rows
  return umma_desc_sw128(img + k16 * 2048, chunk_bytes, 1024);
}

// Load 128 (or 256: global keys) token rows x 128 head columns starting at rolled position pos0 into a two-chunk image.
// Windowed with a shift: row r holds token (pos0 + r + shift) mod Tp.  Only the LAST 128-position block contains the
// wrap (shift < 16 <= window): its rows [0, nmain) are tokens [pos0 + shift, Tp) and rows [nmain, nmain + shift) are
// tokens [0, shift), nmain = Tp - shift - pos0.  The full box goes first (tokens >= T are out of bounds = zeros, which
// also clears every row the block does not own), the wrap rows land on top of it in a second, ordered phase.
// Returns the number of barrier phases used (1 or 2); the caller waits for them in order.
__device__ __forceinline__ int load_rows(uint8_t* dst, int chunk_bytes, const CUtensorMap* mapMain,
                                         const CUtensorMap* mapTail, uint64_t* bar, uint32_t& phase, int col0, int pos0,
                                         int b, int Tp, int shift, int box_bytes) {
  const int t0 = pos0 + shift;
  mbar_arrive_expect_tx(bar, 2 * box_bytes);
  tma_load_3d(dst, mapMain, bar, col0, t0, b);
  tma_load_3d(dst + chunk_bytes, mapMain, bar, col0 + 64, t0, b);
  if (shift > 0 && t0 + 128 > Tp) {                   // this block holds the wrap-around rows
    const int nmain = Tp - t0;
    mbar_wait(bar, phase);                            // the zero-filled rows must be down before the wrap rows land
    phase ^= 1;
    mbar_arrive_expect_tx(bar, 2 * shift * 128);
    tma_load_3d(dst + nmain * 128, mapTail, bar, col0, 0, b);
    tma_load_3d(dst + chunk_bytes + nmain * 128, mapTail, bar, col0 + 64, 0, b);
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// forward.  grid = B * H * nblk.  NKB = number of 128-key blocks in the score tile (1: T <= 128 or windowed, 2).
// ------------------------------------------------------------------------------------------------
template <int NKB>
__global__ void __launch_bounds__(kA2Threads, 1)
attn2_fwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmQtail,
                 const __grid_constant__ CUtensorMap tmKV, const __grid_constant__ Attn2P P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int kKVChunk = NKB * kChunk128;          // bytes of a [NKB*128 rows][64 cols] chunk
  uint8_t* sQ = smem;                                // 32 KB
  uint8_t* sK = sQ + 2 * kChunk128;                  // NKB * 32 KB; P ([128][NKB*128]) aliases it after S
  uint8_t* sV = sK + 2 * kKVChunk;                   // NKB * 32 KB
  float* sBias = reinterpret_cast<float*>(sV + 2 * kKVChunk);        // [512] (2*Prel-1 <= 511), log2 domain
  uint64_t* bars = reinterpret_cast<uint64_t*>(sBias + 512);
  uint64_t* bar_load = bars, *bar_s = bars + 1, *bar_p = bars + 2, *bar_o = bars + 3, *bar_lk = bars + 4, *bar_lv = bars + 5;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qb = blockIdx.x % P.nblk;
  const int bh = blockIdx.x / P.nblk, b = bh / P.H, h = bh - b * P.H;
  const bool windowed = P.window > 0;

  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmKV);
    mbar_init(bar_load, 1); mbar_init(bar_s, 1); mbar_init(bar_p, 128); mbar_init(bar_o, 1);
    mbar_init(bar_lk, 1); mbar_init(bar_lv, 1);
    fence_barrier_init();
  }
  if (warp == 4) tmem_alloc(tmem_slot, 512);
  for (int i = threadIdx.x; i < 512; i += kA2Threads)
    sBias[i] = (P.table && i < 2 * P.Prel - 1) ? P.table[i * P.H + h] * kLog2e : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  constexpr uint32_t idesc_s = umma_idesc_bf16(128, NKB * 128, 0, 0);
  constexpr uint32_t idesc_o = umma_idesc_bf16(128, 128, 0, 1);
  const int D = P.H * kA2Hd;

  if (warp == 4) {
    if (lane == 0) {
      // three independent load barriers (Q, K, V): each may need a second, ordered phase for the wrap-around rows
      uint32_t phq = 0, phk = 0, phv = 0;
      if (windowed) {                                 // keys/values = the same 128 rolled positions as the queries
        load_rows(sQ, kChunk128, &tmQ, &tmQtail, bar_load, phq, h * kA2Hd, qb * 128, b, P.Tp, P.shift, kChunk128);
        load_rows(sK, kKVChunk, &tmQ, &tmQtail, bar_lk, phk, D + h * kA2Hd, qb * 128, b, P.Tp, P.shift, kChunk128);
        load_rows(sV, kKVChunk, &tmQ, &tmQtail, bar_lv, phv, 2 * D + h * kA2Hd, qb * 128, b, P.Tp, P.shift, kChunk128);
      } else {
        load_rows(sQ, kChunk128, &tmQ, &tmQtail, bar_load, phq, h * kA2Hd, qb * 128, b, P.Tp, 0, kChunk128);
        load_rows(sK, kKVChunk, &tmKV, &tmKV, bar_lk, phk, D + h * kA2Hd, 0, b, P.Tp, 0, kKVChunk);
        load_rows(sV, kKVChunk, &tmKV, &tmKV, bar_lv, phv, 2 * D + h * kA2Hd, 0, b, P.Tp, 0, kKVChunk);
      }
      mbar_wait(bar_load, phq);
      mbar_wait(bar_lk, phk);
      mbar_wait(bar_lv, phv);
      tc_fence_after();
      const uint32_t q = smem_u32(sQ), k = smem_u32(sK);
#pragma unroll
      for (int i = 0; i < 8; ++i)
        umma_bf16(tmem, d_kmajor(q, kChunk128, i), d_kmajor(k, kKVChunk, i), idesc_s, i ? 1u : 0u);
      umma_commit(bar_s);
      mbar_wait(bar_p, 0);
      tc_fence_after();
      const uint32_t pp = smem_u32(sK), v = smem_u32(sV);
#pragma unroll
      for (int i = 0; i < NKB * 8; ++i)
        umma_bf16(tmem + 256, d_kmajor(pp, kChunk128, i), d_mnmajor(v, kKVChunk, i), idesc_o, i ? 1u : 0u);
      umma_commit(bar_o);
    }
  } else {
    const int r = warp * 32 + lane;
    const int pi = qb * 128 + r;                                   // rolled position of this query
    int ti = pi + (windowed ? P.shift : 0);
    if (ti >= P.Tp) ti -= P.Tp;
    const bool rok = pi < P.Tp && ti < P.T;                        // a real (not padded) query token
    const uint32_t trow = tmem + (static_cast<uint32_t>(warp * 32) << 16);
    const float sl2 = P.scale * kLog2e;
    const float inv_keep = P.drop_p > 0.f ? 1.0f / (1.0f - P.drop_p) : 1.0f;
    uint8_t* sP = sK;
    mbar_wait(bar_s, 0);
    tc_fence_after();
    float m = -INFINITY, sum = 0.f;
    if (windowed) {
      const int wb = r & ~15, ri = r & 15;
      // tcgen05.ld is warp-collective (one column address per warp): read the warp's 32 diagonal columns, each
      // half-warp keeps its own 16-key window
      uint32_t rawa[16], rawb[16];
      tmem_ld16(trow + warp * 32, rawa);
      tmem_ld16(trow + warp * 32 + 16, rawb);
      tmem_ld_wait();
      const bool upper = (lane & 16) != 0;
      float e[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int pj = qb * 128 + wb + j;
        int tj = pj + P.shift;
        if (tj >= P.Tp) tj -= P.Tp;
        const bool ok = pj < P.Tp && tj < P.T;                     // key padding mask (True = valid), rolled like the tokens
        const float sv = __uint_as_float(upper ? rawb[j] : rawa[j]);
        e[j] = ok ? fmaf(sv, sl2, sBias[j - ri + P.Prel - 1]) : -INFINITY;
        m = fmaxf(m, e[j]);
      }
      if (!rok) m = 0.f;                                           // padded query row: all-zero probabilities, no NaN
#pragma unroll
      for (int j = 0; j < 16; ++j) { e[j] = rok ? ex2f(e[j] - m) : 0.f; sum += e[j]; }
      if (!rok) sum = 1.f;
      if (P.drop_p > 0.f) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          int tj = qb * 128 + wb + j + P.shift;
          if (tj >= P.Tp) tj -= P.Tp;
          e[j] *= attn_keep(P.seed, bh, ti, tj, P.drop_p, inv_keep);
        }
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");               // every row has read its scores: K may be reused
      uint4 lo, hi;
      lo.x = pack_bf16(e[0], e[1]); lo.y = pack_bf16(e[2], e[3]); lo.z = pack_bf16(e[4], e[5]); lo.w = pack_bf16(e[6], e[7]);
      hi.x = pack_bf16(e[8], e[9]); hi.y = pack_bf16(e[10], e[11]); hi.z = pack_bf16(e[12], e[13]); hi.w = pack_bf16(e[14], e[15]);
      const uint4 z = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
      for (int g = 0; g < 16; ++g) {
        const uint4 v = (g == (wb >> 3)) ? lo : ((g == (wb >> 3) + 1) ? hi : z);
        store_row8(sP, kChunk128, r, g >> 3, g & 7, v);
      }
    } else {
      // pass 1: row maximum over all keys
#pragma unroll 1
      for (int c = 0; c < NKB * 128; c += 16) {
        uint32_t raw[16];
        tmem_ld16(trow + c, raw);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int pj = c + j;
          if (pj < P.T) m = fmaxf(m, fmaf(__uint_as_float(raw[j]), sl2, sBias[max(pj - pi + P.Prel - 1, 0)]));
        }
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");               // (second pass re-reads TMEM, not the K image)
      // pass 2: exponentials, row sum, P image (overwrites K: all rows passed the barrier only after the S MMA,
      // which is the last reader of K)
#pragma unroll 1
      for (int c = 0; c < NKB * 128; c += 16) {
        uint32_t raw[16];
        tmem_ld16(trow + c, raw);
        tmem_ld_wait();
        float e[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int pj = c + j;
          e[j] = pj < P.T ? ex2f(fmaf(__uint_as_float(raw[j]), sl2, sBias[max(pj - pi + P.Prel - 1, 0)]) - m) : 0.f;
          sum += e[j];
          if (P.drop_p > 0.f) e[j] *= attn_keep(P.seed, bh, ti, pj, P.drop_p, inv_keep);
        }
        uint4 lo, hi;
        lo.x = pack_bf16(e[0], e[1]); lo.y = pack_bf16(e[2], e[3]); lo.z = pack_bf16(e[4], e[5]); lo.w = pack_bf16(e[6], e[7]);
        hi.x = pack_bf16(e[8], e[9]); hi.y = pack_bf16(e[10], e[11]); hi.z = pack_bf16(e[12], e[13]); hi.w = pack_bf16(e[14], e[15]);
        const int g = c >> 3;
        store_row8(sP, kChunk128, r, g >> 3, g & 7, lo);
        store_row8(sP, kChunk128, r, (g + 1) >> 3, (g + 1) & 7, hi);
      }
    }
    const float inv = __fdividef(1.0f, sum);
    fence_proxy_async();
    tc_fence_before();
    mbar_arrive(bar_p);
    if (rok && P.lse) P.lse[static_cast<long long>(bh) * P.T + ti] = (m + lg2f(sum)) * kLn2;
    mbar_wait(bar_o, 0);
    tc_fence_after();
    __nv_bfloat16* orow = P.out + (static_cast<long long>(b) * P.T + ti) * D + h * kA2Hd;
#pragma unroll
    for (int c = 0; c < 128; c += 16) {
      uint32_t raw[16];
      tmem_ld16(trow + 256 + c, raw);
      tmem_ld_wait();
      if (rok) {
        uint4 u0, u1;
        u0.x = pack_bf16(__uint_as_float(raw[0]) * inv, __uint_as_float(raw[1]) * inv);
        u0.y = pack_bf16(__uint_as_float(raw[2]) * inv, __uint_as_float(raw[3]) * inv);
        u0.z = pack_bf16(__uint_as_float(raw[4]) * inv, __uint_as_float(raw[5]) * inv);
        u0.w = pack_bf16(__uint_as_float(raw[6]) * inv, __uint_as_float(raw[7]) * inv);
        u1.x = pack_bf16(__uint_as_float(raw[8]) * inv, __uint_as_float(raw[9]) * inv);
        u1.y = pack_bf16(__uint_as_float(raw[10]) * inv, __uint_as_float(raw[11]) * inv);
        u1.z = pack_bf16(__uint_as_float(raw[12]) * inv, __uint_as_float(raw[13]) * inv);
        u1.w = pack_bf16(__uint_as_float(raw[14]) * inv, __uint_as_float(raw[15]) * inv);
        *reinterpret_cast<uint4*>(orow + c) = u0;
        *reinterpret_cast<uint4*>(orow + c + 8) = u1;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------------------------------------
// backward.  grid = B * H * nblk: CTA (b, h, key block kb) loops over the query blocks that attend to it.
// TMEM columns: [0,128) S then dQ, [128,256) dP, [256,384) dK (accumulated), [384,512) dV (accumulated)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kA2Threads, 1)
attn2_bwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmQtail,
                 const __grid_constant__ CUtensorMap tmDO, const __grid_constant__ CUtensorMap tmDOtail,
                 const __grid_constant__ Attn2P P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sK = smem + 2 * kChunk128;
  uint8_t* sV = smem + 4 * kChunk128;
  uint8_t* sDO = smem + 6 * kChunk128;
  uint8_t* sP = smem + 8 * kChunk128;
  uint8_t* sDS = smem + 10 * kChunk128;
  float* sBias = reinterpret_cast<float*>(smem + 12 * kChunk128);     // [512] natural-log domain * log2e
  float* sDB = sBias + 512;                                           // [512] bias-gradient bins
  uint64_t* bars = reinterpret_cast<uint64_t*>(sDB + 512);
  uint64_t* bar_kv = bars, *bar_q = bars + 1, *bar_s = bars + 2, *bar_p = bars + 3, *bar_g = bars + 4, *bar_free = bars + 5;
  uint64_t* bar_v = bars + 6, *bar_do = bars + 7;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kb = blockIdx.x % P.nblk;
  const int bh = blockIdx.x / P.nblk, b = bh / P.H, h = bh - b * P.H;
  const bool windowed = P.window > 0;
  const int shift = windowed ? P.shift : 0;
  const int q_first = windowed ? kb : 0, q_count = windowed ? 1 : P.nblk;

  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmDO);
    mbar_init(bar_kv, 1); mbar_init(bar_q, 1); mbar_init(bar_s, 1); mbar_init(bar_p, 128); mbar_init(bar_g, 1);
    mbar_init(bar_free, 128); mbar_init(bar_v, 1); mbar_init(bar_do, 1);
    fence_barrier_init();
  }
  if (warp == 4) tmem_alloc(tmem_slot, 512);
  for (int i = threadIdx.x; i < 512; i += kA2Threads) {
    sBias[i] = (P.table && i < 2 * P.Prel - 1) ? P.table[i * P.H + h] * kLog2e : 0.f;
    sDB[i] = 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  constexpr uint32_t id_kk = umma_idesc_bf16(128, 128, 0, 0);
  constexpr uint32_t id_km = umma_idesc_bf16(128, 128, 0, 1);
  constexpr uint32_t id_mm = umma_idesc_bf16(128, 128, 1, 1);
  const int D = P.H * kA2Hd;

  if (warp == 4) {
    if (lane == 0) {
      uint32_t phk = 0, phv = 0, phq = 0, phdo = 0;    // running phases of the four load barriers
      load_rows(sK, kChunk128, &tmQ, &tmQtail, bar_kv, phk, D + h * kA2Hd, kb * 128, b, P.Tp, shift, kChunk128);
      load_rows(sV, kChunk128, &tmQ, &tmQtail, bar_v, phv, 2 * D + h * kA2Hd, kb * 128, b, P.Tp, shift, kChunk128);
      const uint32_t q = smem_u32(sQ), k = smem_u32(sK), v = smem_u32(sV), d_o = smem_u32(sDO);
      const uint32_t pp = smem_u32(sP), ds = smem_u32(sDS);
      for (int it = 0; it < q_count; ++it) {
        const int qb = q_first + it;
        const uint32_t ph = it & 1;
        if (it > 0) mbar_wait(bar_free, ph ^ 1);                  // previous dQ read out, Q / dO / P / dS images free
        load_rows(sQ, kChunk128, &tmQ, &tmQtail, bar_q, phq, h * kA2Hd, qb * 128, b, P.Tp, shift, kChunk128);
        load_rows(sDO, kChunk128, &tmDO, &tmDOtail, bar_do, phdo, h * kA2Hd, qb * 128, b, P.Tp, shift, kChunk128);
        if (it == 0) { mbar_wait(bar_kv, phk); mbar_wait(bar_v, phv); }
        mbar_wait(bar_q, phq); phq ^= 1;
        mbar_wait(bar_do, phdo); phdo ^= 1;
        tc_fence_after();
#pragma unroll
        for (int i = 0; i < 8; ++i)
          umma_bf16(tmem, d_kmajor(q, kChunk128, i), d_kmajor(k, kChunk128, i), id_kk, i ? 1u : 0u);            // S
#pragma unroll
        for (int i = 0; i < 8; ++i)
          umma_bf16(tmem + 128, d_kmajor(d_o, kChunk128, i), d_kmajor(v, kChunk128, i), id_kk, i ? 1u : 0u);    // dP
        umma_commit(bar_s);
        mbar_wait(bar_p, ph);
        tc_fence_after();
        const uint32_t acc = it > 0 ? 1u : 0u;
#pragma unroll
        for (int i = 0; i < 8; ++i)
          umma_bf16(tmem + 384, d_mnmajor(pp, kChunk128, i), d_mnmajor(d_o, kChunk128, i), id_mm, (i ? 1u : 0u) | acc);  // dV += P^T dO
#pragma unroll
        for (int i = 0; i < 8; ++i)
          umma_bf16(tmem + 256, d_mnmajor(ds, kChunk128, i), d_mnmajor(q, kChunk128, i), id_mm, (i ? 1u : 0u) | acc);    // dK += dS^T Q
#pragma unroll
        for (int i = 0; i < 8; ++i)
          umma_bf16(tmem, d_kmajor(ds, kChunk128, i), d_mnmajor(k, kChunk128, i), id_km, i ? 1u : 0u);                   // dQ = dS K
        umma_commit(bar_g);
      }
    }
  } else {
    const int r = warp * 32 + lane;
    const uint32_t trow = tmem + (static_cast<uint32_t>(warp * 32) << 16);
    const float sl2 = P.scale * kLog2e;
    const float inv_keep = P.drop_p > 0.f ? 1.0f / (1.0f - P.drop_p) : 1.0f;
    for (int it = 0; it < q_count; ++it) {
      const int qb = q_first + it;
      const uint32_t ph = it & 1;
      const int pi = qb * 128 + r;
      int ti = pi + shift;
      if (ti >= P.Tp) ti -= P.Tp;
      const bool rok = pi < P.Tp && ti < P.T;
      float delta = 0.f;
      if (rok) {
        const uint4* po = reinterpret_cast<const uint4*>(P.o + (static_cast<long long>(b) * P.T + ti) * D + h * kA2Hd);
        const uint4* pd = reinterpret_cast<const uint4*>(P.dout + (static_cast<long long>(b) * P.T + ti) * D + h * kA2Hd);
#pragma unroll 4
        for (int i = 0; i < 16; ++i) {
          const uint4 a = __ldg(po + i), c = __ldg(pd + i);
          float2 x, y;
          x = unpack_bf16(a.x); y = unpack_bf16(c.x); delta += x.x * y.x + x.y * y.y;
          x = unpack_bf16(a.y); y = unpack_bf16(c.y); delta += x.x * y.x + x.y * y.y;
          x = unpack_bf16(a.z); y = unpack_bf16(c.z); delta += x.x * y.x + x.y * y.y;
          x = unpack_bf16(a.w); y = unpack_bf16(c.w); delta += x.x * y.x + x.y * y.y;
        }
      }
      const float lse2 = rok ? P.lse[static_cast<long long>(bh) * P.T + ti] * kLog2e : 0.f;
      mbar_wait(bar_s, ph);
      tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < 128; c += 16) {
        // windowed: only the two 16-key chunks on this warp's diagonal carry data (warp-uniform test: tcgen05.ld
        // is warp-collective); within them a lane keeps the chunk that is its own window
        const bool live = !windowed || ((c >> 5) == warp);
        const bool mine = !windowed || (c == (r & ~15));
        float p[16], ds[16];
        if (live) {
          uint32_t rs[16], rp[16];
          tmem_ld16(trow + c, rs);
          tmem_ld16(trow + 128 + c, rp);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int pj = kb * 128 + c + j;
            int tkey = pj + shift;
            if (tkey >= P.Tp) tkey -= P.Tp;
            const bool ok = rok && mine && pj < P.Tp && tkey < P.T;
            const int bidx = max(pj - pi + P.Prel - 1, 0);
            const float pr = ok ? ex2f(fmaf(__uint_as_float(rs[j]), sl2, sBias[bidx]) - lse2) : 0.f;
            float keep = 1.f;
            if (P.drop_p > 0.f && ok) {
              keep = attn_keep(P.seed, bh, ti, tkey, P.drop_p, inv_keep);
            }
            const float dsr = pr * (__uint_as_float(rp[j]) * keep - delta);    // d(score incl. bias)
            p[j] = pr * keep;
            ds[j] = dsr * P.scale;
            if (P.dtable && ok) atomicAdd(&sDB[bidx], dsr);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) { p[j] = 0.f; ds[j] = 0.f; }
        }
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          uint4 u, w;
          u.x = pack_bf16(p[8 * g], p[8 * g + 1]); u.y = pack_bf16(p[8 * g + 2], p[8 * g + 3]);
          u.z = pack_bf16(p[8 * g + 4], p[8 * g + 5]); u.w = pack_bf16(p[8 * g + 6], p[8 * g + 7]);
          w.x = pack_bf16(ds[8 * g], ds[8 * g + 1]); w.y = pack_bf16(ds[8 * g + 2], ds[8 * g + 3]);
          w.z = pack_bf16(ds[8 * g + 4], ds[8 * g + 5]); w.w = pack_bf16(ds[8 * g + 6], ds[8 * g + 7]);
          const int gg = (c >> 3) + g;
          store_row8(sP, kChunk128, r, gg >> 3, gg & 7, u);
          store_row8(sDS, kChunk128, r, gg >> 3, gg & 7, w);
        }
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(bar_p);
      mbar_wait(bar_g, ph);
      tc_fence_after();
      // dQ rows of this query block
      __nv_bfloat16* dst;
      if (q_count == 1 || P.nblk == 1) dst = P.dqkv + (static_cast<long long>(b) * P.T + ti) * (3 * D) + h * kA2Hd;
      else dst = P.dq_part + ((static_cast<long long>(kb) * P.B + b) * P.T + ti) * D + h * kA2Hd;
#pragma unroll 1
      for (int c = 0; c < 128; c += 16) {
        uint32_t raw[16];
        tmem_ld16(trow + c, raw);
        tmem_ld_wait();
        if (rok) {
          uint4 u0, u1;
          u0.x = pack_bf16(__uint_as_float(raw[0]), __uint_as_float(raw[1]));
          u0.y = pack_bf16(__uint_as_float(raw[2]), __uint_as_float(raw[3]));
          u0.z = pack_bf16(__uint_as_float(raw[4]), __uint_as_float(raw[5]));
          u0.w = pack_bf16(__uint_as_float(raw[6]), __uint_as_float(raw[7]));
          u1.x = pack_bf16(__uint_as_float(raw[8]), __uint_as_float(raw[9]));
          u1.y = pack_bf16(__uint_as_float(raw[10]), __uint_as_float(raw[11]));
          u1.z = pack_bf16(__uint_as_float(raw[12]), __uint_as_float(raw[13]));
          u1.w = pack_bf16(__uint_as_float(raw[14]), __uint_as_float(raw[15]));
          *reinterpret_cast<uint4*>(dst + c) = u0;
          *reinterpret_cast<uint4*>(dst + c + 8) = u1;
        }
      }
      tc_fence_before();
      mbar_arrive(bar_free);
    }
    // dK, dV rows of this key block (token of key row r)
    {
      const int pj = kb * 128 + r;
      int tj = pj + shift;
      if (tj >= P.Tp) tj -= P.Tp;
      const bool kok = pj < P.Tp && tj < P.T;
      __nv_bfloat16* base = P.dqkv + (static_cast<long long>(b) * P.T + tj) * (3 * D) + h * kA2Hd;
      const uint32_t cols[2] = {256u, 384u};           // dK, dV
#pragma unroll 1
      for (int w = 0; w < 2; ++w) {
        __nv_bfloat16* dst = base + (w + 1) * D;
#pragma unroll 1
        for (int c = 0; c < 128; c += 16) {
          uint32_t raw[16];
          tmem_ld16(trow + cols[w] + c, raw);
          tmem_ld_wait();
          if (kok) {
            uint4 u0, u1;
            u0.x = pack_bf16(__uint_as_float(raw[0]), __uint_as_float(raw[1]));
            u0.y = pack_bf16(__uint_as_float(raw[2]), __uint_as_float(raw[3]));
            u0.z = pack_bf16(__uint_as_float(raw[4]), __uint_as_float(raw[5]));
            u0.w = pack_bf16(__uint_as_float(raw[6]), __uint_as_float(raw[7]));
            u1.x = pack_bf16(__uint_as_float(raw[8]), __uint_as_float(raw[9]));
            u1.y = pack_bf16(__uint_as_float(raw[10]), __uint_as_float(raw[11]));
            u1.z = pack_bf16(__uint_as_float(raw[12]), __uint_as_float(raw[13]));
            u1.w = pack_bf16(__uint_as_float(raw[14]), __uint_as_float(raw[15]));
            *reinterpret_cast<uint4*>(dst + c) = u0;
            *reinterpret_cast<uint4*>(dst + c + 8) = u1;
          }
        }
      }
    }
    if (P.dtable) {
      asm volatile("bar.sync 1, 128;" ::: "memory");
      for (int i = r; i < 2 * P.Prel - 1; i += 128) {
        const float v = sDB[i];
        if (v != 0.f) atomicAdd(P.dtable + static_cast<long long>(i) * P.H + h, v);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem, 512);
}

// dqkv[:, :, 0, :, :] = sum over key blocks of the partial dQ          (global attention with T > 128)
__global__ void add_dq_kernel(const __nv_bfloat16* __restrict__ part, int nblk, long long rows, int D,
                              __nv_bfloat16* __restrict__ dqkv) {
  const long long n8 = rows * D / 8;
  const int G = D / 8;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n8;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long row = i / G;
    const int g = static_cast<int>(i - row * G);
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int k = 0; k < nblk; ++k) {
      const uint4 u = *reinterpret_cast<const uint4*>(part + (static_cast<long long>(k) * rows + row) * D + g * 8);
      float2 t;
      t = unpack_bf16(u.x); acc[0] += t.x; acc[1] += t.y;
      t = unpack_bf16(u.y); acc[2] += t.x; acc[3] += t.y;
      t = unpack_bf16(u.z); acc[4] += t.x; acc[5] += t.y;
      t = unpack_bf16(u.w); acc[6] += t.x; acc[7] += t.y;
    }
    uint4 o;
    o.x = pack_bf16(acc[0], acc[1]); o.y = pack_bf16(acc[2], acc[3]);
    o.z = pack_bf16(acc[4], acc[5]); o.w = pack_bf16(acc[6], acc[7]);
    *reinterpret_cast<uint4*>(dqkv + row * (3LL * D) + g * 8) = o;
  }
}

}  // namespace htrvt

using namespace htrvt;

namespace {
typedef CUresult (*EncodeTiledFn2)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn2 attn2_encode() {
  static EncodeTiledFn2 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn2>(p);
  }
  return fn;
}
// 3-D map (cols, rows, z), box {64, box_rows, 1}, SWIZZLE_128B
int a2_map3(CUtensorMap* m, const void* ptr, long long cols, long long rows, long long z, long long row_stride,
            long long z_stride, int box_rows) {
  EncodeTiledFn2 enc = attn2_encode();
  if (!enc) return HTRVT_ERR_DRIVER;
  if (reinterpret_cast<uintptr_t>(ptr) & 15) return HTRVT_ERR_ALIGN;
  cuuint64_t gd[3] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows), static_cast<cuuint64_t>(z)};
  cuuint64_t gs[2] = {static_cast<cuuint64_t>(row_stride) * 2, static_cast<cuuint64_t>(z_stride) * 2};
  cuuint32_t bx[3] = {64, static_cast<cuuint32_t>(box_rows), 1}, es[3] = {1, 1, 1};
  if ((gs[0] & 15) || (gs[1] & 15)) return HTRVT_ERR_ALIGN;
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), gd, gs, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? HTRVT_OK : HTRVT_ERR_DRIVER;
}

}  // namespace

int htrvt::attention2_check(int B, int H, int T, int hd, int window, int shift, int Prel, const void* table) {
  if (hd != kA2Hd || T < 1 || T > 256 || B < 1 || H < 1) return HTRVT_ERR_SHAPE;
  if (window != 0 && window != 16) return HTRVT_ERR_SHAPE;
  if (window == 0 && shift != 0) return HTRVT_ERR_SHAPE;
  if (window && (shift < 0 || shift >= window || (shift % 8))) return HTRVT_ERR_SHAPE;   // any T <= 256: padded + masked
  if (table && (Prel < T || 2 * Prel - 1 > 511)) return HTRVT_ERR_SHAPE;
  if (!table && Prel != 0 && Prel < T) return HTRVT_ERR_SHAPE;
  return HTRVT_OK;
}

// Attention with relative-position bias, global (window = 0) or 16-token windows over the sequence rolled by
// -shift (model_window/model/HTR_VT.py:33-62, 114-154).  qkv bf16 token-major [B][T][3*H*128]; out bf16
// [B][T][H*128]; lse fp32 [B][H][T]; table fp32 [2*Prel-1][H] (nullable: no bias); drop_p / seed: attention dropout.
extern "C" int htrvt_attention2_fwd(const void* qkv, int B, int H, int T, int hd, float scale, const float* table,
                                    int Prel, int window, int shift, float drop_p, unsigned long long seed, void* out,
                                    float* lse, cudaStream_t stream) {
  int r = attention2_check(B, H, T, hd, window, shift, Prel, table);
  if (r) return r;
  if (!(drop_p >= 0.f && drop_p < 1.f)) return HTRVT_ERR_SHAPE;     // (also refuses NaN)
  if (!table) Prel = 256;
  const long long ld = 3LL * H * kA2Hd;
  const int nblk = (T + 127) / 128;
  const int nkb = window ? 1 : nblk;
  CUtensorMap tq, tqt, tkv;
  r = a2_map3(&tq, qkv, ld, T, B, ld, static_cast<long long>(T) * ld, 128);
  if (r) return r;
  r = a2_map3(&tqt, qkv, ld, T, B, ld, static_cast<long long>(T) * ld, shift > 0 ? shift : 8);
  if (r) return r;
  r = a2_map3(&tkv, qkv, ld, T, B, ld, static_cast<long long>(T) * ld, nkb * 128);
  if (r) return r;
  Attn2P P = {};
  P.B = B; P.H = H; P.T = T; P.Tp = window ? (T + window - 1) / window * window : T; P.nblk = nblk; P.window = window; P.shift = shift; P.Prel = Prel; P.scale = scale;
  P.table = table; P.out = static_cast<__nv_bfloat16*>(out); P.lse = lse; P.drop_p = drop_p; P.seed = seed;
  const int smem = 2 * kChunk128 + 4 * nkb * kChunk128 + 2048 + 128 + 1024;
  auto kern = nkb == 1 ? attn2_fwd_kernel<1> : attn2_fwd_kernel<2>;
  if (!(nkb == 1 ? HTRVT_ENSURE_SMEM(attn2_fwd_kernel<1>, smem) : HTRVT_ENSURE_SMEM(attn2_fwd_kernel<2>, smem)))
    return HTRVT_ERR_LAUNCH;
  kern<<<B * H * nblk, kA2Threads, smem, stream>>>(tq, tqt, tkv, P);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

extern "C" size_t htrvt_attention2_bwd_workspace_bytes(int B, int H, int T, int window) {
  const int nblk = (T + 127) / 128;
  return (window == 0 && nblk > 1) ? static_cast<size_t>(nblk) * B * T * H * kA2Hd * 2 : 0;
}

// dqkv bf16 [B][T][3][H][128]; dtable fp32 [2*Prel-1][H] (+=, nullable); workspace: partial dQ (see above)
extern "C" int htrvt_attention2_bwd(const void* qkv, const void* out, const void* dout, const float* lse, int B, int H,
                                    int T, int hd, float scale, const float* table, int Prel, int window, int shift,
                                    float drop_p, unsigned long long seed, void* dqkv, float* dtable, void* workspace,
                                    size_t workspace_bytes, cudaStream_t stream) {
  int r = attention2_check(B, H, T, hd, window, shift, Prel, table);
  if (r) return r;
  if (!lse || !(drop_p >= 0.f && drop_p < 1.f)) return HTRVT_ERR_SHAPE;
  if (!table) { Prel = 256; dtable = nullptr; }
  const long long ld = 3LL * H * kA2Hd, ldo = static_cast<long long>(H) * kA2Hd;
  const int nblk = (T + 127) / 128;
  const size_t need = htrvt_attention2_bwd_workspace_bytes(B, H, T, window);
  if (need && (!workspace || workspace_bytes < need)) return HTRVT_ERR_WORKSPACE;
  CUtensorMap tq, tqt, tdo, tdot;
  r = a2_map3(&tq, qkv, ld, T, B, ld, static_cast<long long>(T) * ld, 128);
  if (r) return r;
  r = a2_map3(&tqt, qkv, ld, T, B, ld, static_cast<long long>(T) * ld, shift > 0 ? shift : 8);
  if (r) return r;
  r = a2_map3(&tdo, dout, ldo, T, B, ldo, static_cast<long long>(T) * ldo, 128);
  if (r) return r;
  r = a2_map3(&tdot, dout, ldo, T, B, ldo, static_cast<long long>(T) * ldo, shift > 0 ? shift : 8);
  if (r) return r;
  Attn2P P = {};
  P.B = B; P.H = H; P.T = T; P.Tp = window ? (T + window - 1) / window * window : T; P.nblk = nblk;
  P.window = window; P.shift = shift; P.Prel = Prel; P.scale = scale;
  P.table = table; P.dtable = dtable; P.lse = const_cast<float*>(lse);
  P.o = static_cast<const __nv_bfloat16*>(out); P.dout = static_cast<const __nv_bfloat16*>(dout);
  P.dqkv = static_cast<__nv_bfloat16*>(dqkv); P.dq_part = static_cast<__nv_bfloat16*>(workspace);
  P.drop_p = drop_p; P.seed = seed;
  const int smem = 12 * kChunk128 + 4096 + 128 + 1024;
  if (!HTRVT_ENSURE_SMEM(attn2_bwd_kernel, smem)) return HTRVT_ERR_LAUNCH;
  attn2_bwd_kernel<<<B * H * nblk, kA2Threads, smem, stream>>>(tq, tqt, tdo, tdot, P);
  HTRVT_LAUNCH_CHECK();
  if (need) {
    const long long rows = static_cast<long long>(B) * T;
    const long long n8 = rows * ldo / 8;
    const int blocks = static_cast<int>((n8 + 255) / 256 < 148 * 8 ? (n8 + 255) / 256 : 148 * 8);
    add_dq_kernel<<<blocks, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(workspace), nblk, rows,
                                             static_cast<int>(ldo), static_cast<__nv_bfloat16*>(dqkv));
    HTRVT_LAUNCH_CHECK();
  }
  return HTRVT_OK;
}
