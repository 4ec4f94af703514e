// fp32-parity mode of the eval-mode encoder ("precision = fp32"): every tensor between kernels is fp32, every dense
// contraction still runs on the tcgen05 tap GEMM, fed with SPLIT-bf16 operands: x = h + m + l with h = bf16(x),
// m = bf16(x - h), l = bf16(x - h - m) (3 x 8 mantissa bits = fp32's 24), and
//   x . w  ~=  h.h' + h.m' + m.h' + m.m' + h.l' + l.h'          (dropped terms <= 2^-24 relative)
// as six accumulating launches into an fp32 output (bf16 x bf16 products are exact in the fp32 accumulator).
// The kernels here are the fp32 element-wise / normalisation / attention steps between those GEMMs; each writes the
// fp32 result (kept for residual adds) and, where the next consumer is a GEMM, its three bf16 planes.
// Purpose: logits within 1e-4 of the fp32 reference (model_v1/model/HTR_VT.py:222-241 run by torch in fp32) and greedy
// decode strings identical to the reference's end to end (north_star).  Not a throughput path: ~6x the GEMM time.
#include "common.cuh"

namespace htrvt {

__device__ __forceinline__ void split3(float x, __nv_bfloat16& h, __nv_bfloat16& m, __nv_bfloat16& l) {
  h = __float2bfloat16_rn(x);
  const float r1 = x - __bfloat162float(h);          // exact (Sterbenz-like: h is x rounded to 8 bits)
  m = __float2bfloat16_rn(r1);
  const float r2 = r1 - __bfloat162float(m);         // exact
  l = __float2bfloat16_rn(r2);
}

// planes[3][n] <- split(src[n])
__global__ void split3_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ planes, long long n) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    __nv_bfloat16 h, m, l;
    split3(src[i], h, m, l);
    planes[i] = h; planes[n + i] = m; planes[2 * n + i] = l;
  }
}

// y = [relu](raw * scale[c] + shift[c] [+ res | + raw2 * scale2[c] + shift2[c]]) on fp32 NHWC tensors [P][C];
// y (nullable) fp32, planes (nullable) bf16 [3][P*C]
__global__ void bn_act_f32_kernel(const float* __restrict__ raw, const float* __restrict__ scale,
                                  const float* __restrict__ shift, const float* __restrict__ res,
                                  const float* __restrict__ raw2, const float* __restrict__ scale2,
                                  const float* __restrict__ shift2, float* __restrict__ y,
                                  __nv_bfloat16* __restrict__ planes, long long n, int C, int relu) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    float v = scale ? fmaf(raw[i], scale[c], shift[c]) : raw[i];
    if (res) v += res[i];
    else if (raw2) v += fmaf(raw2[i], scale2[c], shift2[c]);
    if (relu) v = fmaxf(v, 0.f);
    if (y) y[i] = v;
    if (planes) {
      __nv_bfloat16 h, m, l;
      split3(v, h, m, l);
      planes[i] = h; planes[n + i] = m; planes[2 * n + i] = l;
    }
  }
}

// MaxPool2d(3, stride (2,1), pad 1) on fp32 NHWC [B,H,W,C] -> [B,Ho,W,C]
__global__ void maxpool_f32_kernel(const float* __restrict__ in, float* __restrict__ out, int B, int H, int W, int C) {
  const int Ho = (H - 1) / 2 + 1;
  const long long n = static_cast<long long>(B) * Ho * W * C;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    long long r = i / C;
    const int wo = static_cast<int>(r % W); r /= W;
    const int ho = static_cast<int>(r % Ho);
    const int b = static_cast<int>(r / Ho);
    float best = -INFINITY;
    for (int kh = 0; kh < 3; ++kh) {
      const int hh = 2 * ho + kh - 1;
      if (hh < 0 || hh >= H) continue;
      for (int kw = 0; kw < 3; ++kw) {
        const int ww = wo + kw - 1;
        if (ww < 0 || ww >= W) continue;
        best = fmaxf(best, in[((static_cast<long long>(b) * H + hh) * W + ww) * C + c]);
      }
    }
    out[i] = best;
  }
}

// x[b,t,:] = (mask ? tok * m + (1 - m) * mask_token : tok) + pos[t,:]          (all fp32)
__global__ void tokens_f32_kernel(const float* __restrict__ tok, const float* __restrict__ mask,
                                  const float* __restrict__ mask_token, const float* __restrict__ pos,
                                  float* __restrict__ x, int B, int T, int D) {
  const long long n = static_cast<long long>(B) * T * D;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int d = static_cast<int>(i % D);
    const int t = static_cast<int>((i / D) % T);
    float v = tok[i];
    if (mask) { const float m = mask[t]; v = v * m + (1.f - m) * mask_token[d]; }
    if (pos) v += pos[static_cast<long long>(t) * D + d];
    x[i] = v;
  }
}

// row LayerNorm (affine, eps) of x (+ addend) in fp32: one warp per row.  x_out (nullable) = x + addend;
// planes bf16 [3][M*D] (nullable) / y fp32 (nullable) = LN(x + addend)
__global__ void __launch_bounds__(256) row_ln_f32_kernel(const float* __restrict__ x, const float* __restrict__ addend,
                                                         float* __restrict__ x_out, const float* __restrict__ gamma,
                                                         const float* __restrict__ beta, float* __restrict__ y,
                                                         __nv_bfloat16* __restrict__ planes, int M, int D, float eps) {
  const int lane = threadIdx.x & 31;
  const long long n = static_cast<long long>(M) * D;
  for (int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < M; row += gridDim.x * (blockDim.x >> 5)) {
    const float* xr = x + static_cast<long long>(row) * D;
    const float* ar = addend ? addend + static_cast<long long>(row) * D : nullptr;
    float s = 0.f;
    for (int d = lane; d < D; d += 32) s += xr[d] + (ar ? ar[d] : 0.f);
    const float mean = warp_sum(s) / D;
    float q = 0.f;
    for (int d = lane; d < D; d += 32) { const float v = xr[d] + (ar ? ar[d] : 0.f) - mean; q = fmaf(v, v, q); }
    const float rstd = 1.0f / sqrtf(warp_sum(q) / D + eps);
    for (int d = lane; d < D; d += 32) {
      const float v = xr[d] + (ar ? ar[d] : 0.f);
      const long long o = static_cast<long long>(row) * D + d;
      if (x_out) x_out[o] = v;
      const float z = (v - mean) * rstd * gamma[d] + beta[d];
      if (y) y[o] = z;
      if (planes) {
        __nv_bfloat16 h, m, l;
        split3(z, h, m, l);
        planes[o] = h; planes[n + o] = m; planes[2 * n + o] = l;
      }
    }
  }
}

// planes[3][n] <- split(gelu_erf(u[n]))   (exact erf form: timm Mlp's nn.GELU)
__global__ void gelu_split_kernel(const float* __restrict__ u, __nv_bfloat16* __restrict__ planes, long long n) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float v = u[i];
    const float a = 0.5f * v * (1.0f + erff(v * 0.70710678118654752f));
    __nv_bfloat16 h, m, l;
    split3(a, h, m, l);
    planes[i] = h; planes[n + i] = m; planes[2 * n + i] = l;
  }
}

// softmax(q k^T * scale) v in fp32 (model_v1/model/HTR_VT.py:31-35).  qkv fp32 [B,T,3,H,hd], out fp32 [B,T,H*hd].
// CTA = 32 query rows of one (b, h); 4 lanes per row, each owning hd/4 = 32 of the head dims; keys in tiles of 32
// through shared memory with the usual running max / sum (fp32: the rescaling only reorders roundings).
constexpr int kExHd = 128, kExRows = 32, kExKeys = 32;
__global__ void __launch_bounds__(128) attention_f32_kernel(const float* __restrict__ qkv, float* __restrict__ out, int B,
                                                            int H, int T, float scale) {
  __shared__ float ks[kExKeys][kExHd + 4];
  __shared__ float vs[kExKeys][kExHd + 4];
  const int qblocks = (T + kExRows - 1) / kExRows;
  const int qb = blockIdx.x % qblocks, bh = blockIdx.x / qblocks;
  const int h = bh % H, b = bh / H;
  const int row = qb * kExRows + (threadIdx.x >> 2), part = threadIdx.x & 3;
  const long long tok_stride = 3LL * H * kExHd;
  const float* base = qkv + static_cast<long long>(b) * T * tok_stride + h * kExHd;
  float q[32], o[32];
  const bool ok = row < T;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    q[i] = ok ? base[static_cast<long long>(row) * tok_stride + part * 32 + i] * 1.0f : 0.f;
    o[i] = 0.f;
  }
  float mx = -INFINITY, sum = 0.f;
  for (int k0 = 0; k0 < T; k0 += kExKeys) {
    __syncthreads();
    for (int i = threadIdx.x; i < kExKeys * kExHd; i += blockDim.x) {
      const int kk = i / kExHd, d = i - kk * kExHd;
      const bool kv_ok = k0 + kk < T;
      const float* tp = base + static_cast<long long>(k0 + kk) * tok_stride;
      ks[kk][d] = kv_ok ? tp[H * kExHd + d] : 0.f;
      vs[kk][d] = kv_ok ? tp[2 * H * kExHd + d] : 0.f;
    }
    __syncthreads();
    const int nk = min(kExKeys, T - k0);
    for (int kk = 0; kk < nk; ++kk) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 32; ++i) s = fmaf(q[i], ks[kk][part * 32 + i], s);
      s += __shfl_xor_sync(0xffffffffu, s, 1);
      s += __shfl_xor_sync(0xffffffffu, s, 2);
      s *= scale;
      const float nm = fmaxf(mx, s);
      const float corr = expf(mx - nm), p = expf(s - nm);          // first key: mx = -inf -> corr = 0
      sum = sum * corr + p;
#pragma unroll
      for (int i = 0; i < 32; ++i) o[i] = fmaf(o[i], corr, p * vs[kk][part * 32 + i]);
      mx = nm;
    }
  }
  if (ok) {
    const float inv = 1.0f / sum;
    float* op = out + (static_cast<long long>(b) * T + row) * (H * kExHd) + h * kExHd + part * 32;
#pragma unroll
    for (int i = 0; i < 32; ++i) op[i] = o[i] * inv;
  }
}

// softmax(q k^T * scale + bias) v in fp32 with the windowed variant's semantics (model_window/model/HTR_VT.py:33-62,
// 114-154; htrvt_attention2_fwd is its 16-bit counterpart).  CTA shape, lane split and arithmetic of
// attention_f32_kernel; bias = table[(j - i) + Prel - 1][h], the head's column staged in shared memory.
//   global   (window 0): the CTA's 32 queries scan all T keys in tiles of 32.
//   windowed (window 16): the sequence is zero-padded to Tp = ceil16(T) and rolled by -shift, so rolled position p
//     holds token (p + shift) mod Tp.  A CTA takes 32 consecutive rolled positions = two windows, stages their keys
//     once, and each row reads only the 16 keys of its own window (i, j window-local: the wrap-around window mixes head
//     and tail tokens, as the reference does).  Keys of padded tokens (>= T) are skipped, i.e. weight exactly 0 as
//     the reference's finfo.min fill gives; padded query rows are never stored.  A warp's 8 rows share one window,
//     so the skip is warp-uniform.
__global__ void __launch_bounds__(128) attention2_f32_kernel(const float* __restrict__ qkv, float* __restrict__ out,
                                                             const float* __restrict__ table, int B, int H, int T,
                                                             int Prel, int window, int shift, float scale) {
  __shared__ float ks[kExKeys][kExHd + 4];
  __shared__ float vs[kExKeys][kExHd + 4];
  __shared__ float bias[512];
  const int Tp = window ? (T + window - 1) / window * window : T;
  const int qblocks = (Tp + kExRows - 1) / kExRows;
  const int qb = blockIdx.x % qblocks, bh = blockIdx.x / qblocks;
  const int h = bh % H, b = bh / H;
  const int r = threadIdx.x >> 2, part = threadIdx.x & 3;
  const int pos = qb * kExRows + r;                         // query position (rolled when windowed)
  auto token = [&](int p) { const int t = p + shift; return t >= Tp ? t - Tp : t; };
  const long long tok_stride = 3LL * H * kExHd;
  const float* base = qkv + static_cast<long long>(b) * T * tok_stride + h * kExHd;
  for (int i = threadIdx.x; i < 512; i += blockDim.x) bias[i] = (table && i < 2 * Prel - 1) ? table[i * H + h] : 0.f;
  const int tq = token(pos);
  const bool ok = pos < Tp && tq < T;
  float q[32], o[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    q[i] = ok ? base[static_cast<long long>(tq) * tok_stride + part * 32 + i] * 1.0f : 0.f;
    o[i] = 0.f;
  }
  float mx = -INFINITY, sum = 0.f;
  const int ntiles = window ? 1 : (T + kExKeys - 1) / kExKeys;
  for (int tile = 0; tile < ntiles; ++tile) {
    const int p0 = window ? qb * kExRows : tile * kExKeys;   // first key position of the tile
    __syncthreads();                                         // (also publishes `bias` before the first tile)
    for (int i = threadIdx.x; i < kExKeys * kExHd; i += blockDim.x) {
      const int kk = i / kExHd, d = i - kk * kExHd;
      const int tk = token(p0 + kk);
      const bool kv_ok = p0 + kk < Tp && tk < T;
      const float* tp = base + static_cast<long long>(tk) * tok_stride;
      ks[kk][d] = kv_ok ? tp[H * kExHd + d] : 0.f;
      vs[kk][d] = kv_ok ? tp[2 * H * kExHd + d] : 0.f;
    }
    __syncthreads();
    const int lo = window ? (r & ~15) : 0;
    const int hi = window ? lo + 16 : min(kExKeys, T - p0);
    for (int kk = lo; kk < hi; ++kk) {
      const int p = p0 + kk;
      if (p >= Tp || token(p) >= T) continue;               // padded key (windowed only)
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 32; ++i) s = fmaf(q[i], ks[kk][part * 32 + i], s);
      s += __shfl_xor_sync(0xffffffffu, s, 1);
      s += __shfl_xor_sync(0xffffffffu, s, 2);
      // (q k^T) * scale, then + bias: the reference's two roundings.  The clamp only acts on rows that are never
      // stored (global, pos >= T) and on windowed tables shorter than the window, which the reference cannot build
      s = __fmul_rn(s, scale) + bias[max(p - pos + Prel - 1, 0)];
      const float nm = fmaxf(mx, s);
      const float corr = expf(mx - nm), pr = expf(s - nm);  // first key: mx = -inf -> corr = 0
      sum = sum * corr + pr;
#pragma unroll
      for (int i = 0; i < 32; ++i) o[i] = fmaf(o[i], corr, pr * vs[kk][part * 32 + i]);
      mx = nm;
    }
  }
  if (ok) {
    const float inv = 1.0f / sum;
    float* op = out + (static_cast<long long>(b) * T + tq) * (H * kExHd) + h * kExHd + part * 32;
#pragma unroll
    for (int i = 0; i < 32; ++i) op[i] = o[i] * inv;
  }
}

}  // namespace htrvt

using namespace htrvt;

static inline int ex_grid(long long n, int block) {
  long long g = (n + block - 1) / block;
  return static_cast<int>(g < 1 ? 1 : (g > 148LL * 16 ? 148LL * 16 : g));
}

extern "C" int htrvt_split3(const float* src, void* planes_bf16, long long n, cudaStream_t stream) {
  if (n <= 0 || !src || !planes_bf16) return HTRVT_ERR_SHAPE;
  split3_kernel<<<ex_grid(n, 256), 256, 0, stream>>>(src, static_cast<__nv_bfloat16*>(planes_bf16), n);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

extern "C" int htrvt_bn_act_f32(const float* raw, const float* scale, const float* shift, const float* res,
                                const float* raw2, const float* scale2, const float* shift2, float* y,
                                void* planes_bf16, long long P, int C, int relu, cudaStream_t stream) {
  if (P <= 0 || C <= 0 || !raw) return HTRVT_ERR_SHAPE;
  const long long n = P * C;
  bn_act_f32_kernel<<<ex_grid(n, 256), 256, 0, stream>>>(raw, scale, shift, res, raw2, scale2, shift2, y,
                                                         static_cast<__nv_bfloat16*>(planes_bf16), n, C, relu);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

extern "C" int htrvt_maxpool_f32(const float* in, float* out, int B, int H, int W, int C, cudaStream_t stream) {
  if (B <= 0 || H <= 0 || W <= 0 || C <= 0) return HTRVT_ERR_SHAPE;
  const long long n = static_cast<long long>(B) * ((H - 1) / 2 + 1) * W * C;
  maxpool_f32_kernel<<<ex_grid(n, 256), 256, 0, stream>>>(in, out, B, H, W, C);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

extern "C" int htrvt_tokens_f32(const float* tok, const float* mask, const float* mask_token, const float* pos,
                                float* x, int B, int T, int D, cudaStream_t stream) {
  if (B <= 0 || T <= 0 || D <= 0) return HTRVT_ERR_SHAPE;
  tokens_f32_kernel<<<ex_grid(static_cast<long long>(B) * T * D, 256), 256, 0, stream>>>(tok, mask, mask_token, pos, x,
                                                                                        B, T, D);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

extern "C" int htrvt_row_ln_f32(const float* x, const float* addend, float* x_out, const float* gamma,
                                const float* beta, float* y, void* planes_bf16, int M, int D, float eps,
                                cudaStream_t stream) {
  if (M <= 0 || D <= 0 || !x || !gamma || !beta) return HTRVT_ERR_SHAPE;
  row_ln_f32_kernel<<<ex_grid((static_cast<long long>(M) + 7) / 8, 1), 256, 0, stream>>>(
      x, addend, x_out, gamma, beta, y, static_cast<__nv_bfloat16*>(planes_bf16), M, D, eps);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

extern "C" int htrvt_gelu_split(const float* u, void* planes_bf16, long long n, cudaStream_t stream) {
  if (n <= 0 || !u || !planes_bf16) return HTRVT_ERR_SHAPE;
  gelu_split_kernel<<<ex_grid(n, 256), 256, 0, stream>>>(u, static_cast<__nv_bfloat16*>(planes_bf16), n);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

extern "C" int htrvt_attention_f32(const float* qkv, int B, int H, int T, int hd, float scale, float* out,
                                   cudaStream_t stream) {
  if (B <= 0 || H <= 0 || T <= 0 || hd != kExHd || !qkv || !out) return HTRVT_ERR_SHAPE;
  const int qblocks = (T + kExRows - 1) / kExRows;
  attention_f32_kernel<<<B * H * qblocks, 128, 0, stream>>>(qkv, out, B, H, T, scale);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

extern "C" int htrvt_attention2_f32(const float* qkv, int B, int H, int T, int hd, float scale, const float* table,
                                    int Prel, int window, int shift, float* out, cudaStream_t stream) {
  const int r = attention2_check(B, H, T, hd, window, shift, Prel, table);
  if (r) return r;
  if (!qkv || !out) return HTRVT_ERR_SHAPE;
  if (!table) Prel = 256;                                   // no table: a zero bias column
  const int Tp = window ? (T + window - 1) / window * window : T;
  const int qblocks = (Tp + kExRows - 1) / kExRows;
  attention2_f32_kernel<<<B * H * qblocks, 128, 0, stream>>>(qkv, out, table, B, H, T, Prel, window, shift, scale);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}
