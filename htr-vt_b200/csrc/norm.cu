// HBM-bound normalisation / elementwise kernels of the transformer part (sm_100a):
// whole-sample LayerNorm (input image and logits slab), row LayerNorm fwd/bwd fused with the fp32
// residual stream, span-mask + positional embedding, GELU backward, bias-gradient column sums,
// weight casts.  All vectorised 16-byte accesses, one pass over HBM where the math allows.
//
// Replaces: LayerNorm.forward (model_v1/model/HTR_VT.py:134-136), nn.LayerNorm(768, eps=1e-6)
// (:68,75,169), random_masking + pos_embed add (:212-220,229-231), nn.GELU backward (timm Mlp).
#include "common.cuh"

namespace htrvt {

// ------------------------------------------------------------------------------------------------
// Whole-sample LayerNorm (no affine): y = (x - mean) * rstd over all N elements of a sample
// ------------------------------------------------------------------------------------------------
template <typename OutT>
__global__ void __launch_bounds__(1024) sample_ln_fwd_kernel(const float* __restrict__ x, OutT* __restrict__ y,
                                                             float* __restrict__ mean_out,
                                                             float* __restrict__ rstd_out, int N, float eps) {
  __shared__ float red[40];
  const float* xb = x + static_cast<long long>(blockIdx.x) * N;
  OutT* yb = y + static_cast<long long>(blockIdx.x) * N;
  float s = 0.f;
  for (int i = threadIdx.x * 4; i < N; i += 4096) {
    const float4 v = *reinterpret_cast<const float4*>(xb + i);
    s += (v.x + v.y) + (v.z + v.w);
  }
  const float mean = block_sum(s, red) / N;
  float q = 0.f;
  for (int i = threadIdx.x * 4; i < N; i += 4096) {
    const float4 v = *reinterpret_cast<const float4*>(xb + i);
    const float a = v.x - mean, b = v.y - mean, c = v.z - mean, d = v.w - mean;
    q += (a * a + b * b) + (c * c + d * d);
  }
  const float var = block_sum(q, red) / N;
  const float rstd = rsqrtf(var + eps);
  if (threadIdx.x == 0) {
    if (mean_out) mean_out[blockIdx.x] = mean;
    if (rstd_out) rstd_out[blockIdx.x] = rstd;
  }
  for (int i = threadIdx.x * 4; i < N; i += 4096) {
    const float4 v = *reinterpret_cast<const float4*>(xb + i);
    const float a = (v.x - mean) * rstd, b = (v.y - mean) * rstd, c = (v.z - mean) * rstd, d = (v.w - mean) * rstd;
    if (sizeof(OutT) == 4) {
      *reinterpret_cast<float4*>(reinterpret_cast<float*>(yb) + i) = make_float4(a, b, c, d);
    } else {
      uint2 u;
      u.x = pack_bf16(a, b); u.y = pack_bf16(c, d);
      *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(yb) + i) = u;
    }
  }
}

// dx = rstd * (dy - mean(dy) - y * mean(dy*y)), y = normalised output.  dx is bf16 [rows, ld_out] with
// the sample's N = T*C elements laid out as T rows of C (padded row stride for the head GEMM's TMA).
__global__ void __launch_bounds__(1024) sample_ln_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ y,
                                                             const float* __restrict__ rstd,
                                                             __nv_bfloat16* __restrict__ dx, int N, int C,
                                                             int ld_out) {
  __shared__ float red[40];
  const long long base = static_cast<long long>(blockIdx.x) * N;
  float s1 = 0.f, s2 = 0.f;
  for (int i = threadIdx.x; i < N; i += 1024) {
    const float g = dy[base + i];
    s1 += g;
    s2 += g * y[base + i];
  }
  const float m1 = block_sum(s1, red) / N;
  const float m2 = block_sum(s2, red) / N;
  const float r = rstd[blockIdx.x];
  const int T = N / C;
  __nv_bfloat16* ob = dx + static_cast<long long>(blockIdx.x) * T * ld_out;
  for (int i = threadIdx.x; i < T * ld_out; i += 1024) {
    const int t = i / ld_out, c = i - t * ld_out;
    float v = 0.f;
    if (c < C) v = r * (dy[base + t * C + c] - m1 - y[base + t * C + c] * m2);
    ob[i] = __float2bfloat16_rn(v);
  }
}

// ------------------------------------------------------------------------------------------------
// Row LayerNorm with affine (D % 128 == 0, D <= 1024): one warp per row
// ------------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(256) row_ln_fwd_kernel(const float* __restrict__ x,
                                                         const __nv_bfloat16* __restrict__ addend,
                                                         float* __restrict__ x_out, const float* __restrict__ gamma,
                                                         const float* __restrict__ beta,
                                                         __nv_bfloat16* __restrict__ y, float* __restrict__ mean_out,
                                                         float* __restrict__ rstd_out, int M, float eps) {
  constexpr int V = D / 128;
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= M) return;
  const float* xr = x + static_cast<long long>(row) * D;
  float4 v[V];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    v[i] = *reinterpret_cast<const float4*>(xr + lane * 4 + 128 * i);
    if (addend) {       // residual stream update fused here: x_out = x + addend (the preceding GEMM's bf16 output)
      const uint2 u = *reinterpret_cast<const uint2*>(addend + static_cast<long long>(row) * D + lane * 4 + 128 * i);
      const float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y);
      v[i].x += a.x; v[i].y += a.y; v[i].z += b.x; v[i].w += b.y;
      *reinterpret_cast<float4*>(x_out + static_cast<long long>(row) * D + lane * 4 + 128 * i) = v[i];
    }
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  const float mean = warp_sum(s) * (1.0f / D);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    q += (a * a + b * b) + (c * c + d * d);
  }
  const float rstd = rsqrtf(warp_sum(q) * (1.0f / D) + eps);
  if (lane == 0) { mean_out[row] = mean; rstd_out[row] = rstd; }
  __nv_bfloat16* yr = y + static_cast<long long>(row) * D;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int c = lane * 4 + 128 * i;
    const float4 g = *reinterpret_cast<const float4*>(gamma + c);
    const float4 b = *reinterpret_cast<const float4*>(beta + c);
    uint2 u;
    u.x = pack_bf16((v[i].x - mean) * rstd * g.x + b.x, (v[i].y - mean) * rstd * g.y + b.y);
    u.y = pack_bf16((v[i].z - mean) * rstd * g.z + b.z, (v[i].w - mean) * rstd * g.w + b.w);
    *reinterpret_cast<uint2*>(yr + c) = u;
  }
}

// gx (+)= rstd * (g*dy - mean(g*dy) - xhat * mean(g*dy*xhat)); per-CTA partial dgamma / dbeta.
// If accumulate == 0 the result overwrites gx (used for the final norm, whose input grad starts the stream).
template <int D>
__global__ void __launch_bounds__(256, D >= 512 ? 2 : 1) row_ln_bwd_kernel(const __nv_bfloat16* __restrict__ dy,
                                                         const float* __restrict__ x, const float* __restrict__ mean,
                                                         const float* __restrict__ rstd,
                                                         const float* __restrict__ gamma, float* __restrict__ gx,
                                                         float* __restrict__ dgamma, float* __restrict__ dbeta, int M,
                                                         int rows_per_cta, int accumulate) {
  constexpr int V = D / 128;
  __shared__ __align__(16) float sg[8][D], sb[8][D];
  float* sgm = &sg[0][0];                                // gamma, read per row from smem instead of living in 4 V
                                                         // registers; aliases the reduction buffer (barrier below)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float4 dg[V], db[V];
#pragma unroll
  for (int i = 0; i < V; ++i) {
    dg[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    db[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (int c = threadIdx.x; c < D; c += 256) sgm[c] = gamma[c];
  __syncthreads();
  const int r0 = blockIdx.x * rows_per_cta;
  const int r1 = min(M, r0 + rows_per_cta);
  for (int row = r0 + warp; row < r1; row += 8) {
    const float mu = mean[row], rs = rstd[row];
    const float* xr = x + static_cast<long long>(row) * D;
    const __nv_bfloat16* dr = dy + static_cast<long long>(row) * D;
    float4 xh[V], gy[V];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < V; ++i) {
      const int c = lane * 4 + 128 * i;
      const float4 xv = *reinterpret_cast<const float4*>(xr + c);
      const uint2 u = *reinterpret_cast<const uint2*>(dr + c);
      const float2 d01 = unpack_bf16(u.x), d23 = unpack_bf16(u.y);
      xh[i] = make_float4((xv.x - mu) * rs, (xv.y - mu) * rs, (xv.z - mu) * rs, (xv.w - mu) * rs);
      dg[i].x += d01.x * xh[i].x; dg[i].y += d01.y * xh[i].y; dg[i].z += d23.x * xh[i].z; dg[i].w += d23.y * xh[i].w;
      db[i].x += d01.x; db[i].y += d01.y; db[i].z += d23.x; db[i].w += d23.y;
      const float4 gmv = *reinterpret_cast<const float4*>(sgm + c);
      gy[i] = make_float4(d01.x * gmv.x, d01.y * gmv.y, d23.x * gmv.z, d23.y * gmv.w);
      s1 += (gy[i].x + gy[i].y) + (gy[i].z + gy[i].w);
      s2 += (gy[i].x * xh[i].x + gy[i].y * xh[i].y) + (gy[i].z * xh[i].z + gy[i].w * xh[i].w);
    }
    const float m1 = warp_sum(s1) * (1.0f / D), m2 = warp_sum(s2) * (1.0f / D);
    float* gr = gx + static_cast<long long>(row) * D;
#pragma unroll
    for (int i = 0; i < V; ++i) {
      const int c = lane * 4 + 128 * i;
      float4 o = make_float4(rs * (gy[i].x - m1 - xh[i].x * m2), rs * (gy[i].y - m1 - xh[i].y * m2),
                             rs * (gy[i].z - m1 - xh[i].z * m2), rs * (gy[i].w - m1 - xh[i].w * m2));
      if (accumulate) {
        const float4 old = *reinterpret_cast<const float4*>(gr + c);
        o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w;
      }
      *reinterpret_cast<float4*>(gr + c) = o;
    }
  }
  __syncthreads();                                       // every warp is done with gamma (sgm aliases sg[0])
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int c = lane * 4 + 128 * i;
    *reinterpret_cast<float4*>(&sg[warp][c]) = dg[i];
    *reinterpret_cast<float4*>(&sb[warp][c]) = db[i];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < D; c += 256) {
    float a = 0.f, b = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) { a += sg[w][c]; b += sb[w][c]; }
    // one fp32 atomic per CTA and column straight into the gradients (no partial buffer, no finalise launch; the
    // order of the additions per column is not fixed)
    atomicAdd(dgamma + c, a);
    atomicAdd(dbeta + c, b);
  }
}

// out[c] (+)= sum_r partial[r*stride + c]  (deterministic second stage of every column reduction)
__global__ void colsum_finalize_kernel(const float* __restrict__ partial, int R, long long stride, int Ccols,
                                       float* __restrict__ out, int accumulate) {
  __shared__ float sh[8][32];                           // block = 32 columns x 8 row lanes
  const int c = blockIdx.x * 32 + (threadIdx.x & 31), lr = threadIdx.x >> 5;
  float s = 0.f;
  if (c < Ccols)
    for (int r = lr; r < R; r += 8) s += partial[r * stride + c];
  sh[lr][threadIdx.x & 31] = s;
  __syncthreads();
  if (lr != 0 || c >= Ccols) return;
  s = 0.f;
  for (int k = 0; k < 8; ++k) s += sh[k][threadIdx.x];
  out[c] = accumulate ? out[c] + s : s;
}

// ------------------------------------------------------------------------------------------------
// tokens: x = (mask ? tok : mask_token) + pos      (fp32 residual stream from the bf16 stem output)
// ------------------------------------------------------------------------------------------------
template <bool F16>
__global__ void tokens_fwd_kernel(const __nv_bfloat16* __restrict__ tok, const float* __restrict__ mask,
                                  const float* __restrict__ mask_token, const float* __restrict__ pos,
                                  float* __restrict__ x, int B, int T, int D) {
  const long long n4 = static_cast<long long>(B) * T * D / 4;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long e = i * 4;
    const int d = static_cast<int>(e % D);
    const int t = static_cast<int>((e / D) % T);
    const uint2 u = *reinterpret_cast<const uint2*>(tok + e);
    float2 a = F16 ? unpack_f16(u.x) : unpack_bf16(u.x), b = F16 ? unpack_f16(u.y) : unpack_bf16(u.y);
    float4 v = make_float4(a.x, a.y, b.x, b.y);
    if (mask) {
      const float m = mask[t];
      const float4 mt = *reinterpret_cast<const float4*>(mask_token + d);
      v.x = v.x * m + (1.f - m) * mt.x; v.y = v.y * m + (1.f - m) * mt.y;
      v.z = v.z * m + (1.f - m) * mt.z; v.w = v.w * m + (1.f - m) * mt.w;
    }
    if (pos) {
      const float4 p = *reinterpret_cast<const float4*>(pos + static_cast<long long>(t) * D + d);
      v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
    }
    *reinterpret_cast<float4*>(x + e) = v;
  }
}

// dtok = gx * mask (bf16); partial[t][d] = sum_b gx[b,t,d] * (1 - mask[t])   (one CTA per token position)
__global__ void __launch_bounds__(256) tokens_bwd_kernel(const float* __restrict__ gx, const float* __restrict__ mask,
                                                         __nv_bfloat16* __restrict__ dtok,
                                                         float* __restrict__ partial, int B, int T, int D) {
  const int t = blockIdx.x;
  const float m = mask ? mask[t] : 1.f;
  for (int d = threadIdx.x; d < D; d += 256) {
    float acc = 0.f;
    for (int b = 0; b < B; ++b) {
      const long long e = (static_cast<long long>(b) * T + t) * D + d;
      const float g = gx[e];
      dtok[e] = __float2bfloat16_rn(g * m);
      acc += g * (1.f - m);
    }
    if (partial) partial[static_cast<long long>(t) * D + d] = acc;
  }
}

// ------------------------------------------------------------------------------------------------
// GELU backward: du = da * (Phi(u) + u phi(u)), erf form (nn.GELU default)
// ------------------------------------------------------------------------------------------------
// (gelu_parts / gelu_val / gelu_grad live in common.cuh: the GEMM epilogues use them too)
__device__ __forceinline__ uint32_t gelu2(uint32_t w) {
  const float2 y = unpack_bf16(w);
  return pack_bf16(gelu_val(y.x), gelu_val(y.y));
}
__device__ __forceinline__ uint32_t gelu_grad2(uint32_t g, uint32_t w) {
  const float2 x = unpack_bf16(g), y = unpack_bf16(w);
  return pack_bf16(x.x * gelu_grad(y.x), x.y * gelu_grad(y.y));
}
// a = gelu(u), erf form (nn.GELU default used by timm Mlp); separate full-occupancy kernel because the GEMM epilogue
// is run by 8 warps only.  Two 16-byte loads in flight per thread.
__global__ void __launch_bounds__(256) gelu_fwd_kernel(const __nv_bfloat16* __restrict__ u, __nv_bfloat16* __restrict__ a,
                                                        long long n8) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n8; i += 2 * stride) {
    const bool two = i + stride < n8;
    const uint4 b0 = *reinterpret_cast<const uint4*>(u + i * 8);
    uint4 b1 = make_uint4(0u, 0u, 0u, 0u);
    if (two) b1 = *reinterpret_cast<const uint4*>(u + (i + stride) * 8);
    uint4 o;
    o.x = gelu2(b0.x); o.y = gelu2(b0.y); o.z = gelu2(b0.z); o.w = gelu2(b0.w);
    *reinterpret_cast<uint4*>(a + i * 8) = o;
    if (two) {
      o.x = gelu2(b1.x); o.y = gelu2(b1.y); o.z = gelu2(b1.z); o.w = gelu2(b1.w);
      *reinterpret_cast<uint4*>(a + (i + stride) * 8) = o;
    }
  }
}

__global__ void __launch_bounds__(256) gelu_bwd_kernel(const __nv_bfloat16* __restrict__ da, const __nv_bfloat16* __restrict__ u,
                                                        __nv_bfloat16* __restrict__ du, long long n8) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n8; i += 2 * stride) {
    const bool two = i + stride < n8;
    const uint4 a0 = *reinterpret_cast<const uint4*>(da + i * 8);
    const uint4 b0 = *reinterpret_cast<const uint4*>(u + i * 8);
    uint4 a1 = make_uint4(0u, 0u, 0u, 0u), b1 = a1;
    if (two) {
      a1 = *reinterpret_cast<const uint4*>(da + (i + stride) * 8);
      b1 = *reinterpret_cast<const uint4*>(u + (i + stride) * 8);
    }
    uint4 o;
    o.x = gelu_grad2(a0.x, b0.x); o.y = gelu_grad2(a0.y, b0.y); o.z = gelu_grad2(a0.z, b0.z); o.w = gelu_grad2(a0.w, b0.w);
    *reinterpret_cast<uint4*>(du + i * 8) = o;
    if (two) {
      o.x = gelu_grad2(a1.x, b1.x); o.y = gelu_grad2(a1.y, b1.y); o.z = gelu_grad2(a1.z, b1.z); o.w = gelu_grad2(a1.w, b1.w);
      *reinterpret_cast<uint4*>(du + (i + stride) * 8) = o;
    }
  }
}

// out = a * b (bf16): the activation backward when gelu'(u) was saved by the forward epilogue and a dropout mask sits
// between the activation and fc2 (model_window: da is masked first, then multiplied)
__global__ void __launch_bounds__(256) mul_bf16_kernel(const __nv_bfloat16* __restrict__ a, const __nv_bfloat16* __restrict__ b,
                                                        __nv_bfloat16* __restrict__ out, long long n8) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n8; i += stride) {
    const uint4 x = *reinterpret_cast<const uint4*>(a + i * 8), y = *reinterpret_cast<const uint4*>(b + i * 8);
    const uint32_t xs[4] = {x.x, x.y, x.z, x.w}, ys[4] = {y.x, y.y, y.z, y.w};
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 p = unpack_bf16(xs[k]), q = unpack_bf16(ys[k]);
      o[k] = pack_bf16(p.x * q.x, p.y * q.y);
    }
    *reinterpret_cast<uint4*>(out + i * 8) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// ------------------------------------------------------------------------------------------------
// Column sums of a bf16 matrix [M, N] (bias gradients): partial[cta][N]
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) colsum_bf16_kernel(const __nv_bfloat16* __restrict__ a, long long ld, int M,
                                                          int N, int rows_per_cta, float* __restrict__ out) {
  // thread handles a pair of columns; blockDim.y row lanes are reduced through shared memory
  __shared__ float2 sm[8][128];
  const int tx = threadIdx.x & 127, ty = threadIdx.x >> 7;       // 128 column pairs x 2 row lanes
  const int r0 = blockIdx.y * rows_per_cta, r1 = min(M, r0 + rows_per_cta);
  const int c = (blockIdx.x * 128 + tx) * 2;
  float2 acc = make_float2(0.f, 0.f);
  if (c < N) {
    for (int r = r0 + ty; r < r1; r += 2) {
      const float2 v = unpack_bf16(*reinterpret_cast<const uint32_t*>(a + r * ld + c));
      acc.x += v.x; acc.y += v.y;
    }
  }
  sm[ty][tx] = acc;
  __syncthreads();
  if (ty == 0 && c < N) {
    const float2 o = sm[1][tx];
    atomicAdd(out + c, acc.x + o.x);                    // out += (one atomic per CTA and column, no finalise launch)
    if (c + 1 < N) atomicAdd(out + c + 1, acc.y + o.y);
  }
}

// ------------------------------------------------------------------------------------------------
// Weight packing (fp32 master -> bf16 operand copies), refreshed every forward because SAM perturbs
// the parameters in place twice per iteration (SURVEY.md 9.19)
// ------------------------------------------------------------------------------------------------
__global__ void cast_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long n) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    dst[i] = __float2bfloat16_rn(src[i]);
}
// dst = bf16(src) for a row-major [M, N] fp32 matrix AND colsum[n] += sum_m dst[m, n] (of the rounded values): the
// residual-stream gradient becomes the bf16 dY of fc2 / proj and their bias gradients in one pass (the separate
// column-sum kernel re-read the bf16 copy).  Thread -> 8 consecutive columns, row lanes strided; N % 8 == 0.
__global__ void __launch_bounds__(256) cast_colsum_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                                          float* __restrict__ colsum, int M, int N, int rows_per_cta) {
  extern __shared__ float cs_sm[];                       // [R][N]
  const int G = N / 8, R = blockDim.x / G;
  const int grp = threadIdx.x % G, lane_r = threadIdx.x / G;
  const int r0 = blockIdx.x * rows_per_cta, r1 = min(M, r0 + rows_per_cta);
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (lane_r < R) {
    for (int r = r0 + lane_r; r < r1; r += 2 * R) {
      float4 v[2][2];
      const bool two = r + R < r1;
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const float* p = src + static_cast<long long>(r + u * R) * N + grp * 8;
        const bool ok = u == 0 || two;
        v[u][0] = ok ? __ldg(reinterpret_cast<const float4*>(p)) : make_float4(0.f, 0.f, 0.f, 0.f);
        v[u][1] = ok ? __ldg(reinterpret_cast<const float4*>(p) + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        if (u == 1 && !two) break;
        uint4 o;
        o.x = pack_bf16(v[u][0].x, v[u][0].y); o.y = pack_bf16(v[u][0].z, v[u][0].w);
        o.z = pack_bf16(v[u][1].x, v[u][1].y); o.w = pack_bf16(v[u][1].z, v[u][1].w);
        *reinterpret_cast<uint4*>(dst + static_cast<long long>(r + u * R) * N + grp * 8) = o;
        float2 t;
        t = unpack_bf16(o.x); acc[0] += t.x; acc[1] += t.y;
        t = unpack_bf16(o.y); acc[2] += t.x; acc[3] += t.y;
        t = unpack_bf16(o.z); acc[4] += t.x; acc[5] += t.y;
        t = unpack_bf16(o.w); acc[6] += t.x; acc[7] += t.y;
      }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) cs_sm[lane_r * N + grp * 8 + k] = acc[k];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < N; c += blockDim.x) {
    float s = 0.f;
    for (int rr = 0; rr < R; ++rr) s += cs_sm[rr * N + c];
    atomicAdd(colsum + c, s);
  }
}
// OIHW fp32 [Cout, Cin, taps] -> bf16 [Cout, taps, Cin]
__global__ void pack_conv_weight_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int Cout,
                                        int Cin, int taps) {
  const long long n = static_cast<long long>(Cout) * Cin * taps;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int ci = static_cast<int>(i % Cin);
    const long long r = i / Cin;
    const int tap = static_cast<int>(r % taps);
    const int co = static_cast<int>(r / taps);
    dst[i] = __float2bfloat16_rn(src[(static_cast<long long>(co) * Cin + ci) * taps + tap]);
  }
}

// All bf16 operand copies of one forward in ONE launch: entry i is a plain cast (taps == 0) or an
// OIHW -> [Cout][taps][Cin] repack.  blockIdx.y = tensor, grid-stride over its elements.
constexpr int kMaxPack = 64;
struct PackTable {
  const float* src[kMaxPack];
  __nv_bfloat16* dst[kMaxPack];
  long long numel[kMaxPack];
  int cin[kMaxPack];
  int taps[kMaxPack];
  const float* scale[kMaxPack];          // conv repack only: per-output-channel factor (BatchNorm folding), or null
  unsigned char f16[kMaxPack];           // destination format: 0 = bf16, 1 = IEEE fp16 (forward conv weights)
};
__device__ __forceinline__ __nv_bfloat16 to16(float v, bool f16) {      // 16-bit pattern carried in a bf16-typed word
  if (!f16) return __float2bfloat16_rn(v);
  const __half h = __float2half_rn(fminf(fmaxf(v, -65504.f), 65504.f));
  return *reinterpret_cast<const __nv_bfloat16*>(&h);
}
__global__ void __launch_bounds__(256) pack_weights_kernel(const __grid_constant__ PackTable T) {
  extern __shared__ float pk_stage[];                   // one output channel's [Cin][taps] block (conv repack)
  const int t = blockIdx.y;
  const float* __restrict__ src = T.src[t];
  __nv_bfloat16* __restrict__ dst = T.dst[t];
  const long long n = T.numel[t];
  const int Cin = T.cin[t], taps = T.taps[t];
  const bool f16 = T.f16[t] != 0;
  if (taps < 0) {
    // transposed cast [R][K] fp32 -> [K][R] bf16 (R = Cin field): OIHW [Cout][Cin*taps] -> [Cin][taps][Cout], the
    // K-major B operand of the input-gradient GEMM.  32 x 32 tiles through smem: both sides contiguous.
    float (*tile)[33] = reinterpret_cast<float (*)[33]>(pk_stage);
    const int R = Cin, K = static_cast<int>(n / R);
    const int tk = (K + 31) / 32, tr = (R + 31) / 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;        // 32 x 8
    for (int tile_id = blockIdx.x; tile_id < tk * tr; tile_id += gridDim.x) {
      const int r0 = (tile_id / tk) * 32, k0 = (tile_id % tk) * 32;
      __syncthreads();
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int r = r0 + ty + 8 * j, k = k0 + tx;
        tile[ty + 8 * j][tx] = (r < R && k < K) ? src[static_cast<long long>(r) * K + k] : 0.f;
      }
      __syncthreads();
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int k = k0 + ty + 8 * j, r = r0 + tx;
        if (r < R && k < K) dst[static_cast<long long>(k) * R + r] = to16(tile[tx][ty + 8 * j], f16);
      }
    }
    return;
  }
  if (taps <= 1) {                                      // plain cast ([out,in] linears, 1x1 convs [Cout][Cin])
    const float* __restrict__ sc1 = T.scale[t];           // 1x1 conv with a folded per-output-channel factor
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x)
      dst[i] = to16(sc1 ? src[i] * sc1[i / Cin] : src[i], f16);
    return;
  }
  // OIHW -> [Cout][taps][Cin]: per output channel a [Cin][taps] -> [taps][Cin] transpose through smem, so both the
  // fp32 read and the bf16 write are contiguous
  const int per = Cin * taps;
  const int Cout = static_cast<int>(n / per);
  const float* __restrict__ sc = T.scale[t];
  for (int co = blockIdx.x; co < Cout; co += gridDim.x) {
    const float f = sc ? sc[co] : 1.0f;
    __syncthreads();
    for (int i = threadIdx.x; i < per; i += blockDim.x) pk_stage[i] = src[static_cast<long long>(co) * per + i];
    __syncthreads();
    for (int i = threadIdx.x; i < per; i += blockDim.x) {
      const int tap = i / Cin, ci = i - tap * Cin;
      dst[static_cast<long long>(co) * per + i] = to16(pk_stage[ci * taps + tap] * f, f16);
    }
  }
}

// In-place inverted dropout (+ per-sample DropPath scale) on a bf16 tensor: x[i] *= keep(seed, site, i) / (1 - p)
// * dp[sample(i)].  The mask is a counter-based hash, so applying the same call to the gradient in the backward
// regenerates it (nothing is stored).  Replaces nn.Dropout / timm DropPath of the windowed variant
// (model_window/model/HTR_VT.py:21-23,59-60,100-110; timm Mlp drop1/drop2) in train mode.
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x85ebca6bu; x ^= x >> 13; x *= 0xc2b2ae35u; x ^= x >> 16;
  return x;
}
__global__ void dropout_bf16_kernel(__nv_bfloat16* __restrict__ x, long long n8, long long per_sample8, float p,
                                    float inv_keep, unsigned long long seed, unsigned site,
                                    const float* __restrict__ dp) {
  const uint32_t key = mix32(static_cast<uint32_t>(seed) ^ (site * 0x9e3779b9u)) ^ static_cast<uint32_t>(seed >> 32);
  const uint32_t thr = static_cast<uint32_t>(p * 16777216.0f);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n8;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float sc = dp ? dp[i / per_sample8] : 1.0f;
    uint4 u = *reinterpret_cast<const uint4*>(x + i * 8);
    uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t r = mix32(key + static_cast<uint32_t>(i) * 4u + k) ^ static_cast<uint32_t>(i >> 30);
      // the two 16-bit halves of one hash decide the two bf16 of this word (keep test at 2^-16 resolution)
      const float2 v = unpack_bf16(w[k]);
      const float k0 = ((r & 0xffffu) << 8) < thr ? 0.f : inv_keep * sc;
      const float k1 = ((r >> 16) << 8) < thr ? 0.f : inv_keep * sc;
      w[k] = pack_bf16(v.x * k0, v.y * k1);
    }
    *reinterpret_cast<uint4*>(x + i * 8) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// in [R][P][C] bf16 (pixels x channels, channels contiguous) -> out [R][C][P] (pixels contiguous): the K-major
// dY^T operand of the weight-gradient GEMM.  64 x 64 tiles through padded smem; grid (ceil(P/64), ceil(C/64), R).
__global__ void __launch_bounds__(256) transpose_px_kernel(const __nv_bfloat16* __restrict__ in,
                                                           __nv_bfloat16* __restrict__ out, int P, int C) {
  __shared__ __align__(16) __nv_bfloat16 tile[64][72];
  const int p0 = blockIdx.x * 64, c0 = blockIdx.y * 64;
  const long long row = blockIdx.z;
  const __nv_bfloat16* src = in + row * P * C;
  __nv_bfloat16* dst = out + row * C * P;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int id = threadIdx.x + 256 * k;
    const int px = id >> 3, cg = id & 7;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (p0 + px < P && c0 + cg * 8 < C)
      v = *reinterpret_cast<const uint4*>(src + static_cast<long long>(p0 + px) * C + c0 + cg * 8);
    *reinterpret_cast<uint4*>(&tile[px][cg * 8]) = v;
  }
  __syncthreads();
  const int ch = threadIdx.x & 63;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int pg = (threadIdx.x >> 6) + 4 * k;
    if (c0 + ch >= C || p0 + pg * 8 >= P) continue;
    uint16_t e[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) e[j] = *reinterpret_cast<const uint16_t*>(&tile[pg * 8 + j][ch]);
    uint4 v;
    v.x = e[0] | (static_cast<uint32_t>(e[1]) << 16); v.y = e[2] | (static_cast<uint32_t>(e[3]) << 16);
    v.z = e[4] | (static_cast<uint32_t>(e[5]) << 16); v.w = e[6] | (static_cast<uint32_t>(e[7]) << 16);
    *reinterpret_cast<uint4*>(dst + static_cast<long long>(c0 + ch) * P + p0 + pg * 8) = v;
  }
}

}  // namespace htrvt

using namespace htrvt;

// in bf16 [R][P][C] -> out bf16 [R][C][P]; P % 8 == 0 and C % 8 == 0
extern "C" int htrvt_transpose_px(const void* in, void* out, long long R, int P, int C, cudaStream_t stream) {
  if (R <= 0 || R > 65535 || P <= 0 || C <= 0 || (P & 7) || (C & 7)) return HTRVT_ERR_SHAPE;
  dim3 grid((P + 63) / 64, (C + 63) / 64, static_cast<unsigned>(R));
  transpose_px_kernel<<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(in),
                                                static_cast<__nv_bfloat16*>(out), P, C);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

static inline int grid_for(long long n, int block) {
  long long g = (n + block - 1) / block;
  return static_cast<int>(g < 1 ? 1 : (g > 148LL * 16 ? 148LL * 16 : g));
}

extern "C" int htrvt_sample_ln_fwd(const float* x, void* y, int y_is_bf16, float* mean, float* rstd, int B, int N,
                                   float eps, cudaStream_t stream) {
  if (B <= 0 || N <= 0 || (N & 3)) return HTRVT_ERR_SHAPE;
  if (y_is_bf16)
    sample_ln_fwd_kernel<__nv_bfloat16><<<B, 1024, 0, stream>>>(x, static_cast<__nv_bfloat16*>(y), mean, rstd, N, eps);
  else
    sample_ln_fwd_kernel<float><<<B, 1024, 0, stream>>>(x, static_cast<float*>(y), mean, rstd, N, eps);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

extern "C" int htrvt_sample_ln_bwd(const float* dy, const float* y, const float* rstd, void* dx_bf16, int B, int N,
                                   int C, int ld_out, cudaStream_t stream) {
  if (B <= 0 || N <= 0 || C <= 0 || (N % C) || ld_out < C) return HTRVT_ERR_SHAPE;
  sample_ln_bwd_kernel<<<B, 1024, 0, stream>>>(dy, y, rstd, static_cast<__nv_bfloat16*>(dx_bf16), N, C, ld_out);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

// y = LN(x [+ addend]); when addend (bf16 [M,D]) is given, x_out (fp32) receives x + addend (may alias x)
extern "C" int htrvt_row_ln_fwd(const float* x, const void* addend_bf16, float* x_out, const float* gamma,
                                const float* beta, void* y_bf16, float* mean, float* rstd, int M, int D, float eps,
                                cudaStream_t stream) {
  if (M <= 0 || (addend_bf16 && !x_out)) return HTRVT_ERR_SHAPE;
  const int grid = (M + 7) / 8;
  const __nv_bfloat16* ad = static_cast<const __nv_bfloat16*>(addend_bf16);
  __nv_bfloat16* yo = static_cast<__nv_bfloat16*>(y_bf16);
  if (D == 768)
    row_ln_fwd_kernel<768><<<grid, 256, 0, stream>>>(x, ad, x_out, gamma, beta, yo, mean, rstd, M, eps);
  else if (D == 128)
    row_ln_fwd_kernel<128><<<grid, 256, 0, stream>>>(x, ad, x_out, gamma, beta, yo, mean, rstd, M, eps);
  else if (D == 256)
    row_ln_fwd_kernel<256><<<grid, 256, 0, stream>>>(x, ad, x_out, gamma, beta, yo, mean, rstd, M, eps);
  else
    return HTRVT_ERR_SHAPE;
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

extern "C" int htrvt_row_ln_bwd_ctas(int M) {
  int ctas = (M + 63) / 64;
  return ctas > 592 ? 592 : ctas;
}

// partial: fp32 [ctas][2][D]; dgamma / dbeta are accumulated (+=)
extern "C" int htrvt_row_ln_bwd(const void* dy_bf16, const float* x, const float* mean, const float* rstd,
                                const float* gamma, float* gx, int accumulate, float* dgamma, float* dbeta,
                                float* partial, int M, int D, cudaStream_t stream) {
  if (M <= 0) return HTRVT_ERR_SHAPE;
  const int ctas = htrvt_row_ln_bwd_ctas(M);
  const int rows = (M + ctas - 1) / ctas;
  const __nv_bfloat16* dy = static_cast<const __nv_bfloat16*>(dy_bf16);
  if (D == 768)
    row_ln_bwd_kernel<768><<<ctas, 256, 0, stream>>>(dy, x, mean, rstd, gamma, gx, dgamma, dbeta, M, rows, accumulate);
  else if (D == 128)
    row_ln_bwd_kernel<128><<<ctas, 256, 0, stream>>>(dy, x, mean, rstd, gamma, gx, dgamma, dbeta, M, rows, accumulate);
  else if (D == 256)
    row_ln_bwd_kernel<256><<<ctas, 256, 0, stream>>>(dy, x, mean, rstd, gamma, gx, dgamma, dbeta, M, rows, accumulate);
  else
    return HTRVT_ERR_SHAPE;
  HTRVT_LAUNCH_CHECK();
  (void)partial;                 // dgamma / dbeta are accumulated (+=) with per-CTA atomics
  return HTRVT_OK;
}

// tok: the stem output, 16-bit [B,T,D] (fp16 when tok_f16, else bf16)
extern "C" int htrvt_tokens_fwd(const void* tok, const float* mask, const float* mask_token, const float* pos,
                                float* x, int B, int T, int D, int tok_f16, cudaStream_t stream) {
  if (B <= 0 || T <= 0 || (D & 3)) return HTRVT_ERR_SHAPE;
  const long long n4 = static_cast<long long>(B) * T * D / 4;
  auto kern = tok_f16 ? tokens_fwd_kernel<true> : tokens_fwd_kernel<false>;
  kern<<<grid_for(n4, 256), 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(tok), mask, mask_token, pos, x, B, T, D);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

// partial: fp32 [T][D] scratch; dmask_token (+=) may be null (no masking => no gradient)
extern "C" int htrvt_tokens_bwd(const float* gx, const float* mask, void* dtok_bf16, float* dmask_token,
                                float* partial, int B, int T, int D, cudaStream_t stream) {
  if (B <= 0 || T <= 0 || D <= 0) return HTRVT_ERR_SHAPE;
  const bool want = mask && dmask_token;
  tokens_bwd_kernel<<<T, 256, 0, stream>>>(gx, mask, static_cast<__nv_bfloat16*>(dtok_bf16), want ? partial : nullptr,
                                           B, T, D);
  HTRVT_LAUNCH_CHECK();
  if (want) {
    colsum_finalize_kernel<<<(D + 31) / 32, 256, 0, stream>>>(partial, T, D, D, dmask_token, 1);
    HTRVT_LAUNCH_CHECK();
  }
  return HTRVT_OK;
}

extern "C" int htrvt_gelu_fwd(const void* u, void* a, long long n, cudaStream_t stream) {
  if (n <= 0 || (n & 7)) return HTRVT_ERR_SHAPE;
  gelu_fwd_kernel<<<grid_for(n / 8, 256), 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(u),
                                                            static_cast<__nv_bfloat16*>(a), n / 8);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

extern "C" int htrvt_gelu_bwd(const void* da, const void* u, void* du, long long n, cudaStream_t stream) {
  if (n <= 0 || (n & 7)) return HTRVT_ERR_SHAPE;
  gelu_bwd_kernel<<<grid_for(n / 8, 256), 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(da),
                                                            static_cast<const __nv_bfloat16*>(u),
                                                            static_cast<__nv_bfloat16*>(du), n / 8);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

extern "C" int htrvt_mul_bf16(const void* a, const void* b, void* out, long long n, cudaStream_t stream) {
  if (n <= 0 || (n & 7)) return HTRVT_ERR_SHAPE;
  mul_bf16_kernel<<<grid_for(n / 8, 256), 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(a),
                                                            static_cast<const __nv_bfloat16*>(b),
                                                            static_cast<__nv_bfloat16*>(out), n / 8);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

extern "C" int htrvt_colsum_rows(int M) {
  int r = (M + 255) / 256;
  return r > 128 ? 128 : r;
}

// out[N] (+)= column sums of a bf16 [M, N] (row stride ld); partial: fp32 [htrvt_colsum_rows(M)][N]
extern "C" int htrvt_colsum_bf16(const void* a, long long ld, int M, int N, float* out, int accumulate,
                                 float* partial, cudaStream_t stream) {
  if (M <= 0 || N <= 0 || (ld & 1)) return HTRVT_ERR_SHAPE;
  const int gy = htrvt_colsum_rows(M);
  const int rows = (M + gy - 1) / gy;
  dim3 grid((N + 255) / 256, gy);
  (void)partial;
  if (!accumulate && cudaMemsetAsync(out, 0, static_cast<size_t>(N) * sizeof(float), stream) != cudaSuccess)
    return HTRVT_ERR_LAUNCH;
  colsum_bf16_kernel<<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(a), ld, M, N, rows, out);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

extern "C" int htrvt_cast_bf16(const float* src, void* dst, long long n, cudaStream_t stream) {
  if (n <= 0) return HTRVT_ERR_SHAPE;
  cast_bf16_kernel<<<grid_for(n, 256), 256, 0, stream>>>(src, static_cast<__nv_bfloat16*>(dst), n);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

// dst bf16 [M, N] = bf16(src fp32 [M, N]); colsum fp32 [N] += column sums of dst (N % 8 == 0, N <= 2048)
extern "C" int htrvt_cast_colsum_bf16(const float* src, void* dst, float* colsum, int M, int N, cudaStream_t stream) {
  if (M <= 0 || N <= 0 || (N & 7) || N > 2048 || !src || !dst || !colsum) return HTRVT_ERR_SHAPE;
  const int G = N / 8;
  const int R = 256 / G;                      // >= 1 for N <= 2048
  const int threads = G * R;
  int ctas = (M + 31) / 32;
  if (ctas > 148 * 8) ctas = 148 * 8;
  const int rows = (M + ctas - 1) / ctas;
  cast_colsum_kernel<<<ctas, threads, static_cast<size_t>(R) * N * sizeof(float), stream>>>(
      src, static_cast<__nv_bfloat16*>(dst), colsum, M, N, rows);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

extern "C" int htrvt_pack_conv_weight(const float* w_oihw, void* dst, int Cout, int Cin, int taps,
                                      cudaStream_t stream) {
  if (Cout <= 0 || Cin <= 0 || taps <= 0) return HTRVT_ERR_SHAPE;
  pack_conv_weight_kernel<<<grid_for(static_cast<long long>(Cout) * Cin * taps, 256), 256, 0, stream>>>(
      w_oihw, static_cast<__nv_bfloat16*>(dst), Cout, Cin, taps);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

// n tensors per call: src fp32, dst bf16, numel elements; scale (nullable array of nullable fp32 [Cout] pointers):
// per-output-channel factor folded into a conv repack (eval-mode BatchNorm folding);
// taps[i] == 0 -> cast, > 0 -> OIHW -> [Cout][taps][Cin],
// < 0 -> transposed cast [cin[i]][numel/cin[i]] -> [numel/cin[i]][cin[i]] (cin[i] = rows of the source matrix)
// f16 (nullable): per-tensor destination format, 0 = bf16, 1 = IEEE fp16 (the forward stem's conv weights)
extern "C" int htrvt_pack_weights(int n, const void* const* src, void* const* dst, const long long* numel,
                                  const int* cin, const int* taps, const void* const* scale, const int* f16,
                                  cudaStream_t stream) {
  if (n <= 0) return HTRVT_OK;
  for (int base = 0; base < n; base += kMaxPack) {
    PackTable T = {};
    const int cnt = n - base < kMaxPack ? n - base : kMaxPack;
    for (int i = 0; i < cnt; ++i) {
      T.src[i] = static_cast<const float*>(src[base + i]);
      T.dst[i] = static_cast<__nv_bfloat16*>(dst[base + i]);
      T.numel[i] = numel[base + i];
      T.cin[i] = cin[base + i] > 0 ? cin[base + i] : 1;
      T.taps[i] = taps[base + i];
      T.scale[i] = scale ? static_cast<const float*>(scale[base + i]) : nullptr;
      T.f16[i] = (f16 && f16[base + i]) ? 1 : 0;
      if (T.scale[i] && T.taps[i] < 1) return HTRVT_ERR_SHAPE;       // folding is wired for the conv repacks only
    }
    int smem = 0;
    for (int i = 0; i < cnt; ++i)
      if (T.taps[i] > 1 && T.cin[i] * T.taps[i] * 4 > smem) smem = T.cin[i] * T.taps[i] * 4;
    for (int i = 0; i < cnt; ++i)
      if (T.taps[i] < 0 && smem < 32 * 33 * 4) smem = 32 * 33 * 4;
    if (smem > 48 * 1024) return HTRVT_ERR_SHAPE;
    dim3 grid(4 * 148, cnt);
    pack_weights_kernel<<<grid, 256, smem, stream>>>(T);
    HTRVT_LAUNCH_CHECK();
  }
  return HTRVT_OK;
}


// x bf16 [n] in place; per_sample = elements per batch sample (DropPath scale dp[b], nullable); n, per_sample % 8 == 0
extern "C" int htrvt_dropout_bf16(void* x, long long n, long long per_sample, float p, unsigned long long seed,
                                  unsigned site, const float* dp, cudaStream_t stream) {
  if (n <= 0 || (n & 7) || per_sample <= 0 || (per_sample & 7) || !(p >= 0.f && p < 1.f)) return HTRVT_ERR_SHAPE;
  const long long n8 = n / 8;
  const int blocks = static_cast<int>((n8 + 255) / 256 < 148 * 16 ? (n8 + 255) / 256 : 148 * 16);
  dropout_bf16_kernel<<<blocks, 256, 0, stream>>>(static_cast<__nv_bfloat16*>(x), n8, per_sample / 8, p,
                                                  1.0f / (1.0f - p), seed, site, dp);
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}
