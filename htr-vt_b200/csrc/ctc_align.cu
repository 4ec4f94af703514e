// CTC forced alignment for sm_100a: the single best alignment (Viterbi path) of a KNOWN transcription through the CTC
// trellis, one warp per line.  The loss kernels (ctc.cu, ctc_grp.cu) sum over the same trellis; this one maximises.
//
// Semantics (restated in float64 by oracle/htrvt_align_oracle.py, which the tests match bit for bit):
//   states s = 0 .. S-1, S = 2L + 1, ext[2k] = 0 (blank), ext[2k+1] = label[k];
//   d_0(0) = lp(0, 0), d_0(1) = lp(0, label[0]), every other state -inf;
//   d_t(s) = m + lp(t, ext[s]), m = max(c0, c1, c2) over c0 = d_{t-1}(s), c1 = d_{t-1}(s-1) (s >= 1),
//            c2 = d_{t-1}(s-2) (s >= 2, ext[s] != 0, ext[s] != ext[s-2]);
//   the back-pointer is the FIRST of c0, c1, c2 equal to m (stay, previous, skip);
//   d is float64: each fp32 input is widened and there is exactly one float64 add per state per frame, after the max;
//   the path ends in S-1 if d(S-1) > d(S-2), else in S-2.
// In logits mode (is_logprob = 0) the recursion runs on the raw logits: every path visits each frame once, so the
// argmax is the one of the log-probs; only the reported scores subtract each frame's log-sum-exp (float64, full row).
//
// Layout: lane i owns states [K i, K i + K) in registers (K from the host's max_target_len hint); the predecessors s-1
// and s-2 of a lane's first states come from the lane below by two shuffles.  Frame t+1's emission gathers are issued
// before frame t's update.  Back-pointers take 2 bits per state, packed into NW = ceil(K / 16) words per lane per frame,
// so a frame is NW coalesced rows of 32 words in the global workspace.  The backtrack is a serial walk of T dependent
// reads: it stages the rows back into shared memory in 4 KB chunks from the end, the next chunk's cp.async in flight
// while the current one is walked, and records the visited state of every frame in the path row.  A final pass over
// the frames, 32 at a time, turns states into classes, writes the frame scores and the span boundaries; each label's
// token score is then the float64 sum of its frames' scores in frame order.
#include "common.cuh"

namespace htrvt {

constexpr int kAlMaxL = 256;               // labels per line (S <= 513), as the lane-group CTC kernel
constexpr int kAlMaxT = 1 << 20;           // frames per line
constexpr int kAlWarps = 4;                // lines per CTA
constexpr int kAlStageWords = 1024;        // one staged chunk of back-pointer rows (4 KB)

struct AlignParams {
  const float* x;                          // [.., C] with element strides sb / st, class axis contiguous
  long long sb, st;
  const int* targets;                      // concatenated (tgt_stride == 0) or padded [B, tgt_stride]; may be null
  const int* input_lengths;                // [B] or null (=> T)
  const int* target_lengths;               // [B]
  int* path;                               // [B, T]
  float* frame_scores;                     // [B, T]
  int* spans;                              // [B, span_stride, 2]
  float* token_scores;                     // [B, span_stride]
  double* score;                           // [B]
  int* status;                             // [B]
  uint32_t* bp;                            // workspace: [B][T][32 NW] back-pointer words
  int B, T, C, is_logprob, tgt_stride, span_stride, lcap;
};

__device__ __forceinline__ void al_cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void al_cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void al_cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// log-sum-exp of one row of logits in float64
__device__ __forceinline__ double al_row_lse(const float* __restrict__ r, int C) {
  float m = -INFINITY;
  for (int c = 0; c < C; ++c) m = fmaxf(m, __ldg(r + c));
  double s = 0.0;
  for (int c = 0; c < C; ++c) s += exp(static_cast<double>(__ldg(r + c)) - static_cast<double>(m));
  return static_cast<double>(m) + log(s);
}

template <int K>
__global__ void __launch_bounds__(kAlWarps * 32) ctc_align_kernel(const AlignParams P) {
  constexpr int NW = (K + 15) / 16;        // back-pointer words per lane per frame
  constexpr int RW = 32 * NW;              // words per frame
  constexpr int CH = kAlStageWords / RW;   // frames per staged chunk (<= 32: one frame per lane when recording)
  constexpr unsigned kFull = 0xffffffffu;
  __shared__ __align__(16) uint32_t stage_all[kAlWarps][2 * kAlStageWords];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int b = blockIdx.x * kAlWarps + wib;
  if (b >= P.B) return;                    // whole warps only
  uint32_t* stage = stage_all[wib];

  const int T = P.T, C = P.C;
  const int Tb = P.input_lengths ? P.input_lengths[b] : T;
  const int L = P.target_lengths[b];
  int* pathb = P.path + static_cast<size_t>(b) * T;
  float* fsb = P.frame_scores + static_cast<size_t>(b) * T;
  int* spb = P.spans + static_cast<size_t>(b) * P.span_stride * 2;
  float* tsb = P.token_scores + static_cast<size_t>(b) * P.span_stride;

  long long toff;                          // where the line's labels start (negative lengths count as 0)
  if (P.tgt_stride > 0) {
    toff = static_cast<long long>(b) * P.tgt_stride;
  } else {
    long long part = 0;
    for (int i = lane; i < b; i += 32) part += max(P.target_lengths[i], 0);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(kFull, part, o);
    toff = part;
  }

  // ---- line checks and labels: status 2 = invalid line data, 1 = infeasible --------------------------------------
  int st = (Tb < 0 || Tb > T || L < 0 || L > P.lcap || (L > 0 && !P.targets)) ? 2 : 0;
  const int S = 2 * L + 1;
  int lab[K];
  unsigned skipm = 0;                      // bit j: state lane K + j may be entered by a skip
  int nrep = 0;
  bool bad = false;
#pragma unroll
  for (int j = 0; j < K; ++j) {
    const int s = lane * K + j;
    lab[j] = 0;
    if (st == 0 && (s & 1) && s < S) {
      const int k = s >> 1;
      const int v = P.targets[toff + k];
      if (v < 1 || v >= C) bad = true;
      else lab[j] = v;
      if (k >= 1) {
        if (P.targets[toff + k - 1] == v) ++nrep;
        else skipm |= 1u << j;
      }
    }
  }
  if (__any_sync(kFull, bad)) st = 2;
  nrep = __reduce_add_sync(kFull, nrep);
  if (st == 0 && Tb < L + nrep) st = 1;

  if (st != 0 || Tb == 0) {                // (Tb == 0 and status 0 imply L == 0: aligned, score 0)
    for (int t = lane; t < T; t += 32) { pathb[t] = -1; fsb[t] = 0.f; }
    for (int k = lane; k < P.span_stride; k += 32) { spb[2 * k] = -1; spb[2 * k + 1] = -1; tsb[k] = 0.f; }
    if (lane == 0) { P.score[b] = st ? -INFINITY : 0.0; P.status[b] = st; }
    return;
  }

  // ---- Viterbi ---------------------------------------------------------------------------------------------------
  const float* xb = P.x + static_cast<long long>(b) * P.sb;
  double d[K];
  float e[K];
#pragma unroll
  for (int j = 0; j < K; ++j) {
    const int s = lane * K + j;
    const float v = __ldg(xb + lab[j]);
    d[j] = (s == 0 || (s == 1 && L > 0)) ? static_cast<double>(v) : -INFINITY;
  }
  if (Tb > 1) {
#pragma unroll
    for (int j = 0; j < K; ++j) e[j] = __ldg(xb + P.st + lab[j]);
  }
  uint32_t* bpl = P.bp + static_cast<size_t>(b) * T * RW;
  for (int t = 1; t < Tb; ++t) {
    float ec[K];
#pragma unroll
    for (int j = 0; j < K; ++j) ec[j] = e[j];
    if (t + 1 < Tb) {
      const float* row = xb + static_cast<long long>(t + 1) * P.st;
#pragma unroll
      for (int j = 0; j < K; ++j) e[j] = __ldg(row + lab[j]);
    }
    double up1 = __shfl_up_sync(kFull, d[K - 1], 1), up2 = __shfl_up_sync(kFull, d[K - 2], 1);
    if (lane == 0) { up1 = -INFINITY; up2 = -INFINITY; }
    uint32_t w[NW];
#pragma unroll
    for (int q = 0; q < NW; ++q) w[q] = 0u;
#pragma unroll
    for (int j = K - 1; j >= 0; --j) {     // descending: d[j-1], d[j-2] still hold frame t-1
      const double c0 = d[j];
      const double c1 = j >= 1 ? d[j >= 1 ? j - 1 : 0] : up1;
      const double c2 = j >= 2 ? d[j >= 2 ? j - 2 : 0] : (j == 1 ? up1 : up2);
      double m = c0;
      uint32_t ch = 0u;
      if (c1 > m) { m = c1; ch = 1u; }
      if (((skipm >> j) & 1u) && c2 > m) { m = c2; ch = 2u; }
      d[j] = m + static_cast<double>(ec[j]);
      w[j >> 4] |= ch << (2 * (j & 15));
    }
#pragma unroll
    for (int q = 0; q < NW; ++q) bpl[static_cast<size_t>(t) * RW + q * 32 + lane] = w[q];
  }

  // ---- end state -------------------------------------------------------------------------------------------------
  double v1 = -INFINITY, v2 = -INFINITY;
#pragma unroll
  for (int j = 0; j < K; ++j) {
    const int s = lane * K + j;
    if (s == S - 1) v1 = d[j];
    if (s == S - 2) v2 = d[j];
  }
  v1 = __shfl_sync(kFull, v1, (S - 1) / K);
  v2 = S >= 2 ? __shfl_sync(kFull, v2, (S - 2) / K) : -INFINITY;
  int s = (S >= 2 && !(v1 > v2)) ? S - 2 : S - 1;
  const double vscore = s == S - 1 ? v1 : v2;

  // ---- backtrack: stage back-pointer rows from the end, record the state of every frame in the path row -----------
  __syncwarp();                            // every lane's back-pointer stores precede the staging reads
  const int cend = (Tb - 1) / CH;
  auto issue = [&](int c, int buf) {
    const uint32_t dst = smem_u32(stage + buf * kAlStageWords);
    const uint32_t* src = bpl + static_cast<size_t>(c) * CH * RW;
    const int n16 = min(CH, Tb - c * CH) * RW / 4;
    for (int i = lane; i < n16; i += 32) al_cp_async16(dst + i * 16, src + i * 4);
    al_cp_commit();
  };
  issue(cend, 0);
  for (int c = cend; c >= 0; --c) {
    const int buf = (cend - c) & 1;
    if (c > 0) {
      issue(c - 1, buf ^ 1);
      al_cp_wait<1>();
    } else {
      al_cp_wait<0>();
    }
    __syncwarp();
    const uint32_t* sw = stage + buf * kAlStageWords;
    const int t0 = c * CH, t1 = min(Tb, t0 + CH) - 1;
    int mine = 0;
    for (int t = t1; t >= t0; --t) {
      if (lane == t - t0) mine = s;
      if (t > 0) {
        const int o = s / K, j = s - o * K;
        const uint32_t wv = sw[(t - t0) * RW + (j >> 4) * 32 + o];
        s -= static_cast<int>((wv >> (2 * (j & 15))) & 3u);
      }
    }
    if (lane < CH && t0 + lane < Tb) pathb[t0 + lane] = mine;
    __syncwarp();                          // the buffer is refilled by the next round's copy
  }

  // ---- states -> classes, frame scores, span boundaries ------------------------------------------------------------
  const int* tg = P.targets + toff;
  double lsum = 0.0;
  int prev_last = -1;                      // state of frame t0 - 1
  for (int t0 = 0; t0 < T; t0 += 32) {
    const int t = t0 + lane;
    const bool live = t < Tb;
    const int sc = live ? pathb[t] : -1;
    int sn = __shfl_down_sync(kFull, sc, 1);
    if (lane == 31) sn = t + 1 < Tb ? pathb[t + 1] : -1;
    int sp = __shfl_up_sync(kFull, sc, 1);
    if (lane == 0) sp = prev_last;
    prev_last = __shfl_sync(kFull, sc, 31);
    __syncwarp();                          // every state of this round is read before any is overwritten
    if (live) {
      const int cls = (sc & 1) ? tg[sc >> 1] : 0;
      const float* xr = xb + static_cast<long long>(t) * P.st;
      const float v = __ldg(xr + cls);
      float fs = v;
      if (!P.is_logprob) {
        const double lse = al_row_lse(xr, C);
        lsum += lse;
        fs = static_cast<float>(static_cast<double>(v) - lse);
      }
      pathb[t] = cls;
      fsb[t] = fs;
      if (sc & 1) {
        const int k = sc >> 1;
        if (sp != sc) spb[2 * k] = t;
        if (sn != sc) spb[2 * k + 1] = t + 1;
      }
    } else if (t < T) {
      pathb[t] = -1;
      fsb[t] = 0.f;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) lsum += __shfl_xor_sync(kFull, lsum, o);
  __syncwarp();                            // spans and frame scores of every lane are visible
  for (int k = lane; k < P.span_stride; k += 32) {
    if (k < L) {
      const int a = spb[2 * k], z = spb[2 * k + 1];
      double acc = 0.0;
      for (int t = a; t < z; ++t) acc += static_cast<double>(fsb[t]);
      tsb[k] = static_cast<float>(acc);
    } else {
      spb[2 * k] = -1;
      spb[2 * k + 1] = -1;
      tsb[k] = 0.f;
    }
  }
  if (lane == 0) {
    P.score[b] = P.is_logprob ? vscore : vscore - lsum;
    P.status[b] = 0;
  }
}

// states per lane for labels up to lmax: S = 2 lmax + 1 <= 32 K
int align_states_per_lane(int lmax) {
  const int S = 2 * lmax + 1;
  return S <= 64 ? 2 : S <= 128 ? 4 : S <= 256 ? 8 : S <= 512 ? 16 : 17;
}

}  // namespace htrvt

using namespace htrvt;

extern "C" size_t htrvt_ctc_align_workspace_bytes(int B, int T, int max_target_len) {
  if (B <= 0 || T <= 0 || T > kAlMaxT || max_target_len > kAlMaxL) return 0;
  const int K = align_states_per_lane(max_target_len < 0 ? kAlMaxL : max_target_len);
  return static_cast<size_t>(B) * T * 32 * ((K + 15) / 16) * sizeof(uint32_t);
}

extern "C" int htrvt_ctc_align(const float* x, long long stride_b, long long stride_t, int is_logprob,
                               const int* targets, int tgt_stride, const int* input_lengths, const int* target_lengths,
                               int B, int T, int C, int max_target_len, int* path, float* frame_scores, int* spans,
                               int span_stride, float* token_scores, double* score, int* status, void* workspace,
                               size_t workspace_bytes, cudaStream_t stream) {
  if (B <= 0 || T <= 0 || T > kAlMaxT || C < 2 || !x || !target_lengths || !path || !frame_scores || !score || !status)
    return HTRVT_ERR_SHAPE;
  if (stride_b < 0 || stride_t < 0 || tgt_stride < 0 || span_stride < 0 || max_target_len > kAlMaxL)
    return HTRVT_ERR_SHAPE;
  if (span_stride > 0 && (!spans || !token_scores)) return HTRVT_ERR_SHAPE;
  const size_t need = htrvt_ctc_align_workspace_bytes(B, T, max_target_len);
  if (!workspace || workspace_bytes < need) return HTRVT_ERR_WORKSPACE;
  if (reinterpret_cast<uintptr_t>(workspace) & 15) return HTRVT_ERR_ALIGN;
  const int lmax = max_target_len < 0 ? kAlMaxL : max_target_len;
  AlignParams P;
  P.x = x; P.sb = stride_b; P.st = stride_t;
  P.targets = targets; P.input_lengths = input_lengths; P.target_lengths = target_lengths;
  P.path = path; P.frame_scores = frame_scores; P.spans = spans; P.token_scores = token_scores;
  P.score = score; P.status = status; P.bp = static_cast<uint32_t*>(workspace);
  P.B = B; P.T = T; P.C = C; P.is_logprob = is_logprob ? 1 : 0; P.tgt_stride = tgt_stride;
  P.span_stride = span_stride;
  P.lcap = min(lmax, span_stride);
  const dim3 grid((B + kAlWarps - 1) / kAlWarps);
  switch (align_states_per_lane(lmax)) {
    case 2: ctc_align_kernel<2><<<grid, kAlWarps * 32, 0, stream>>>(P); break;
    case 4: ctc_align_kernel<4><<<grid, kAlWarps * 32, 0, stream>>>(P); break;
    case 8: ctc_align_kernel<8><<<grid, kAlWarps * 32, 0, stream>>>(P); break;
    case 16: ctc_align_kernel<16><<<grid, kAlWarps * 32, 0, stream>>>(P); break;
    default: ctc_align_kernel<17><<<grid, kAlWarps * 32, 0, stream>>>(P); break;
  }
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}
