/* htrvt.h - C ABI of libhtrvt_b200.so: the sm_100a kernels behind the HTR-VT hot path.
 *
 * The reference (0xk0ry/HTR-VT) is pure Python/PyTorch: its "FFI" for this path is the set of ATen / cuDNN /
 * cuBLAS dispatches issued by model_v1/model/{HTR_VT,resnet18}.py, torch.nn.CTCLoss and
 * CTCLabelConverter.decode.  Each entry point below names the reference call site it replaces
 * (paths relative to the reference root).  INTEGRATION.md shows the ctypes binding a maintainer adds.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch's caching allocator); the library never
 *     allocates or frees device memory and keeps no state besides per-kernel attributes;
 *   - all calls are asynchronous on `stream` (a cudaStream_t passed as void*), re-entrant, no host syncs;
 *   - return value: 0 = ok, -1 bad shape, -2 bad alignment, -3 wrong arch, -4 launch failed,
 *     -5 workspace missing/too small, -6 driver entry point (cuTensorMapEncodeTiled) unavailable;
 *   - "bf16" = __nv_bfloat16; activations of the conv stem are NHWC; matrices are row-major with the stated
 *     leading dimension (elements).  sm_100a only, no CPU fallback.
 */
#ifndef HTRVT_H_
#define HTRVT_H_
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

int htrvt_version(void);
unsigned long long htrvt_launch_count(void); /* kernels launched so far by this library (bench.py gpu_launches) */

/* ---- CTC loss forward-backward -------------------------------------------------------------------------
 * Replaces nn.CTCLoss(reduction='none', zero_infinity=True) as called at model_v1/train.py:27-29 and
 * model_v1/valid.py:36-38 (ATen _ctc_loss + _ctc_loss_backward, blank = 0), optionally fused with the
 * `.log_softmax(2)` of train.py:25 (is_logprob = 0: x are logits and grad is d/d(logits)).
 * x / grad: fp32, class axis contiguous, element strides for the batch and time axes ([B,T,C] or [T,B,C]).
 * targets: int32, concatenated (tgt_stride = 0) or padded [B, tgt_stride]; lengths int32 [B].
 * max_target_len: host-side hint (max label length) or -1 = unknown (worst-case provisioning).
 * nll[b] = 0 and grad = 0 for infeasible samples; grad may be NULL (loss only).
 * grad is scaled by grad_scale[b] (device, may be NULL) or grad_scale_const. */
/* Two kernels serve htrvt_ctc_loss_grad: one CTA per sequence (latency: B up to a few sequences per SM; fp64 linear
 * domain with a log-space fallback) and a group of 4-32 lanes per sequence (throughput: B >= 1024, labels up to 256
 * symbols, fp32 linear domain with a consistency guard); whatever the throughput kernel cannot finish is flagged and
 * redone by the first kernel in a fix-up launch.  htrvt_ctc_set_mode: -1 automatic, 0 CTA-per-sequence only, 1 lane-group
 * kernel at any batch size; returns the previous mode.  htrvt_ctc_flagged_count: sequences the lane-group kernel handed
 * to the fix-up launch since the library was loaded (synchronous read). */
int htrvt_ctc_set_mode(int mode);
long long htrvt_ctc_flagged_count(void);
size_t htrvt_ctc_workspace_bytes(int B, int T, int C, int max_target_len);
int htrvt_ctc_loss_grad(const float* x, long long x_stride_b, long long x_stride_t, int is_logprob,
                        const int* targets, int tgt_stride, const int* input_lengths, const int* target_lengths,
                        int B, int T, int C, int max_target_len, float* nll, float* grad, long long g_stride_b,
                        long long g_stride_t, const float* grad_scale, float grad_scale_const, void* workspace,
                        size_t workspace_bytes, void* stream);
/* The recursion runs in the linear domain on the FP64 pipe; a sequence whose posterior rows fail the
 * sum-to-one / two-sided-likelihood checks (a state flushed below the fp64 range that log space would have kept)
 * is recomputed in log space inside the same launch.  This counts those sequences (synchronous read). */
long long htrvt_ctc_fallback_count(void);

/* ---- greedy CTC decode ---------------------------------------------------------------------------------
 * htrvt_greedy_decode replaces `preds.max(2)` + transpose (model_v1/valid.py:40-41) AND the filtering loop of
 * CTCLabelConverter.decode (model_v1/utils/utils.py:72-86): ids[b, 0:lens[b]] are the kept class ids.
 * htrvt_ctc_collapse takes the already arg-maxed sample-major index stream decode() receives; offsets = int64 [B]
 * exclusive prefix sum of lengths (where each line starts in the stream). */
int htrvt_greedy_decode(const float* logits, long long stride_b, long long stride_t, int B, int T, int C,
                        const int* lengths, int n_character, int* ids, int* lens, int* raw_index, void* stream);
int htrvt_ctc_collapse(const void* index, int index_is_int64, const int* lengths, const long long* offsets, int B,
                       int Tmax, int n_character, int* ids, int* lens, void* stream);

/* ---- K-best CTC alignment paths (LM-rescoring evaluation) ---------------------------------------------------
 * htrvt_ctc_kbest_paths replaces the per-frame beam of `simple_ctc_beam_search_with_lm`
 * (model_window/test_with_kenlm.py:25-51): per frame the K most probable classes extend every beam, the K best
 * (float64 score sums, Python's stable descending order on ties) survive; every surviving path is collapsed
 * (blanks and repeats dropped, :44-51).  One warp per line.  log_probs fp32 through element strides (class axis
 * contiguous); ids int32 [B, K, T] zero padded, lens int32 [B, K] (-1: fewer than K paths exist), scores float64
 * [B, K], beams in the reference's final order.  K <= 8, C <= 256.  id -> char and the language model stay on the
 * host (htr-vt_b200/beam.py). */
int htrvt_ctc_kbest_paths(const float* log_probs, long long stride_b, long long stride_t, const int* lengths, int B,
                          int T, int C, int K, int* ids, int* lens, double* scores, void* stream);

/* ---- CTC prefix beam search (SURVEY.md 8(f) row 4: the search that replaces the toy per-frame beam) --------
 * htrvt_ctc_prefix_beam ranks LABELLINGS where htrvt_ctc_kbest_paths (the reference's
 * `simple_ctc_beam_search_with_lm`, model_window/test_with_kenlm.py:25-59) ranks alignment paths: every beam entry
 * is a collapsed prefix with the summed probability of all its alignments (blank-ending / label-ending parts, float64
 * log space); per frame every entry stays or is extended by every label, an extension that spells an entry of the
 * beam is added to that entry, the K most probable survive (ties: stay entries by rank, then extensions by parent
 * rank and label).  Same buffers as htrvt_ctc_kbest_paths: ids int32 [B, K, T] zero padded, lens int32 [B, K]
 * (-1: fewer than K prefixes exist), scores float64 [B, K] best first.  K <= 16, C <= 256, T * K < 65535. */
int htrvt_ctc_prefix_beam(const float* log_probs, long long stride_b, long long stride_t, const int* lengths, int B,
                          int T, int C, int K, int* ids, int* lens, double* scores, void* stream);

/* ---- CTC prefix beam search with a fused character n-gram LM ----------------------------------------------------
 * htrvt_ctc_prefix_beam_lm is htrvt_ctc_prefix_beam with the language-model term inside the search (Hannun et al.
 * 2014, "First-Pass Large Vocabulary Continuous Speech Recognition using Bi-Directional Recurrent DNNs", algorithm 1),
 * extending the LM evaluation of model_window/test_with_kenlm.py:25-59, where the LM only picks among K finished
 * candidates.  Every beam entry keeps its CTC masses (pb, pnb) exactly as the plain search and a float64 lm = sum over
 * its labels of alpha * ln10 * S + beta, S = log10 p(label | previous order-1 tokens, starting from <s>) by ARPA
 * backoff: the listed prob of (context, w), else bow(context) (0 if unlisted) + log10 p(w | context minus its oldest
 * token), with <unk>'s unigram prob when w has none; S is the float64 sum of the float32 table values, longest
 * context's bow first, found prob last.  Candidates rank by lae(pb', pnb') + lm' (ties as in the plain search); an
 * extension that spells an entry merges its CTC mass into it (lm unchanged).  At the end each survivor's key gains
 * alpha * ln10 * log10 p(</s> | context) (KenLM's score(bos=True, eos=True)) and the survivors are re-ranked stably.
 * alpha = beta = 0 gives the ids, lens and scores of htrvt_ctc_prefix_beam bit for bit.
 * lm_table: lm_slots (a power of two) 32-byte slots {u64 lo, hi; float log10 p, log10 bow; u64 pad}, 32-byte aligned,
 * open addressing with linear probing and at least one empty slot (the layout htr-vt_b200/lm.py packs); lm_order 1..8;
 * token ids <unk> = 0, <s> = 1, </s> = 2; tok_map int32 [n_tok_map]: class id -> token id (ids beyond: <unk>).
 * scores float64 [B, K] = the fused score with the </s> term, ctc_scores float64 [B, K] = lae(pb, pnb), entries in
 * fused order; ids / lens as htrvt_ctc_prefix_beam.  HTRVT_ERR_SHAPE: non-finite alpha or beta, lm_order outside
 * 1..8, a slot count that is not a power of two, or the limits of htrvt_ctc_prefix_beam (K <= 16, C <= 256,
 * T * K < 65535). */
int htrvt_ctc_prefix_beam_lm(const float* log_probs, long long stride_b, long long stride_t, const int* lengths, int B,
                             int T, int C, int K, const void* lm_table, long long lm_slots, int lm_order,
                             const int* tok_map, int n_tok_map, double alpha, double beta, int* ids, int* lens,
                             double* scores, double* ctc_scores, void* stream);

/* ---- CTC prefix beam search constrained to a word lexicon --------------------------------------------------------
 * htrvt_ctc_prefix_beam_lex is htrvt_ctc_prefix_beam (lm_table == nullptr; alpha = beta = 0) or
 * htrvt_ctc_prefix_beam_lm (the same LM arguments) in which every word of the output comes from a word list (Scheidl
 * et al. 2018, "Word Beam Search", "Words" mode).  Classes split into word characters (is_word[c] != 0) and free
 * characters (all others, ids >= n_class_map included).  A labelling is accepted when every maximal run of word
 * characters in it is a lexicon word.  Each entry carries a trie node, 0 = between words: between words a free
 * character stays at 0 and a word character c moves to child(root, c); inside a word at node n a word character c
 * moves to child(n, c) and a free character is allowed only if n ends a word (back to 0); a missing child is not
 * allowed; a stay never changes the node.  In a line's last frame no candidate that leaves its entry at a node that
 * does not end a word is eligible, so the survivors are the K best accepted labellings (lens -1 for all K when none
 * exists; a line of zero frames gives the empty labelling).  Ranking, ties and scores are those of the plain / LM
 * search: the lexicon only removes candidates, and with no word character the results equal theirs bit for bit.
 * Trie in CSR form: first int32 [n_nodes + 1] (node 0 = root), label / child int32 [first[n_nodes]] (the edges of
 * node n are first[n] .. first[n + 1] - 1, sorted by label, child ids < n_nodes), word_end uint8 [n_nodes]; its
 * consistency is the caller's contract (htr-vt_b200/lexicon.py packs and checks it), not re-checked on the device.
 * ctc_scores = lae(pb, pnb), scores = the LM's fused score (= ctc_scores without an LM).  HTRVT_ERR_SHAPE: a null
 * trie array, n_nodes < 1, n_class_map > 0 with no is_word, alpha or beta != 0 without an LM, the LM checks of
 * htrvt_ctc_prefix_beam_lm with one, or the limits of htrvt_ctc_prefix_beam (K <= 16, C <= 256, T * K < 65535). */
int htrvt_ctc_prefix_beam_lex(const float* log_probs, long long stride_b, long long stride_t, const int* lengths, int B,
                              int T, int C, int K, const int* first, const int* label, const int* child,
                              const unsigned char* word_end, int n_nodes, const unsigned char* is_word,
                              int n_class_map, const void* lm_table, long long lm_slots, int lm_order,
                              const int* tok_map, int n_tok_map, double alpha, double beta, int* ids, int* lens,
                              double* scores, double* ctc_scores, void* stream);

/* ---- CTC prefix beam search constrained to a word lexicon, with a fused word n-gram LM -------------------------
 * htrvt_ctc_prefix_beam_lex_wlm is htrvt_ctc_prefix_beam_lex (same trie arguments, same constraint) whose LM scores
 * WORDS (Scheidl et al. 2018, "Word Beam Search", "NGrams" mode): the tokens of a labelling are its maximal runs of
 * word characters; free characters are no tokens.  For words w_1 .. w_m the fused score is
 * lae(pb, pnb) + sum_i [alpha * ln10 * log10 p(w_i | <s> w_1 .. w_i-1) + beta] + alpha * ln10 * log10 p(</s> | <s>
 * w_1 .. w_m), ARPA backoff as htrvt_ctc_prefix_beam_lm.  An entry inside a word at trie node n ranks with
 * alpha * ln10 * smear[n] added (no such term between words); the returned scores carry no smear term, and the
 * survivors are re-ranked stably by them.  lm_table as htrvt_ctc_prefix_beam_lm with 21-bit key fields (token + 1,
 * three per 64-bit word: lo fields 0-2, hi fields 3-5; the layout htr-vt_b200/wordlm.py packs), lm_order 1..6;
 * token ids <unk> = 0, <s> = 1, </s> = 2; node_tok int32 [n_nodes]: the token of the word ending at each node (read
 * at word ends only); smear float32 [n_nodes]: the largest unigram log10 prob of the lexicon words that start with
 * the node's prefix.  ids / lens / scores / ctc_scores as htrvt_ctc_prefix_beam_lex.  HTRVT_ERR_SHAPE: a null trie
 * array, node_tok or smear, n_nodes < 1, non-finite alpha or beta, lm_order outside 1..6, a slot count that is not a
 * power of two, or the limits of htrvt_ctc_prefix_beam (K <= 16, C <= 256, T * K < 65535). */
int htrvt_ctc_prefix_beam_lex_wlm(const float* log_probs, long long stride_b, long long stride_t, const int* lengths,
                                  int B, int T, int C, int K, const int* first, const int* label, const int* child,
                                  const unsigned char* word_end, int n_nodes, const unsigned char* is_word,
                                  int n_class_map, const void* lm_table, long long lm_slots, int lm_order,
                                  const int* node_tok, const float* smear, double alpha, double beta, int* ids,
                                  int* lens, double* scores, double* ctc_scores, void* stream);

/* ---- CTC forced alignment of a known transcription -----------------------------------------------------------
 * htrvt_ctc_align: the single best path (Viterbi) through the CTC trellis of each line's labels, blank = 0, with the
 * frames each label occupies: the alignment torchaudio.functional.forced_align computes one line at a time on the host.
 * States S = 2L + 1, ext[2k] = 0, ext[2k+1] = label[k]; d_0(0) = lp(0, 0), d_0(1) = lp(0, label[0]), others -inf;
 * d_t(s) = max(c0, c1, c2) + lp(t, ext[s]) over c0 = d_{t-1}(s), c1 = d_{t-1}(s-1), c2 = d_{t-1}(s-2) (only when
 * ext[s] != 0 and ext[s] != ext[s-2]); on a tie the FIRST of c0, c1, c2 wins (stay, previous, skip).  d is float64:
 * each fp32 input is widened, one float64 add per state per frame after the max.  The path ends in S-1 if
 * d(S-1) > d(S-2), else in S-2 (a tie ends on the last label); L = 0 gives an all-blank path.
 * x: fp32 log-probs, or raw logits with is_logprob = 0 (the path is the same; the scores below subtract each frame's
 * float64 log-sum-exp over the full row), class axis contiguous, element strides for the batch and time axes.
 * targets / tgt_stride / input_lengths / target_lengths as htrvt_ctc_loss_grad (concatenated: line b's labels start at
 * the sum of the earlier lines' lengths, negative ones counted as 0; input_lengths NULL = T for every line).
 * Outputs for line b with T_b frames:
 *   path int32 [B, T]: the class of every frame t < T_b, -1 beyond;  frame_scores fp32 [B, T]: log-prob of that class at
 *   that frame, 0 beyond;  spans int32 [B, span_stride, 2]: [start, end) frames of label k (the frames spent in state
 *   2k+1), -1 for k >= L;  token_scores fp32 [B, span_stride]: float64 sum of the span's frame scores in frame order,
 *   0 for k >= L;  score float64 [B]: the Viterbi log-prob;  status int32 [B]:
 *     0 aligned (T_b = 0 with L = 0: score 0);
 *     1 infeasible, T_b < L + number of adjacent equal labels: score -inf, path and spans -1;
 *     2 invalid line data: a label outside [1, C), a negative length, T_b > T, L > 256, L > max_target_len (when given)
 *       or L > span_stride, or L > 0 with targets NULL: score -inf, path and spans -1.  Nothing outside the line is read.
 * max_target_len: host-side hint (longest label) or -1 = unknown (worst case, 256); it picks the states per lane and
 * the workspace.  Limits: L <= 256, T <= 2^20.  workspace: htrvt_ctc_align_workspace_bytes(B, T, max_target_len) bytes,
 * 16-byte aligned (back-pointers, B * T * 128 bytes, twice that for a hint above 255 or -1).  spans / token_scores may be
 * NULL when span_stride = 0.  HTRVT_ERR_SHAPE: B <= 0, T <= 0 or above the limit, C < 2, negative strides,
 * max_target_len > 256, a missing output; HTRVT_ERR_WORKSPACE; HTRVT_ERR_ALIGN.  Deterministic, no atomics. */
size_t htrvt_ctc_align_workspace_bytes(int B, int T, int max_target_len);
int htrvt_ctc_align(const float* x, long long stride_b, long long stride_t, int is_logprob, const int* targets,
                    int tgt_stride, const int* input_lengths, const int* target_lengths, int B, int T, int C,
                    int max_target_len, int* path, float* frame_scores, int* spans, int span_stride,
                    float* token_scores, double* score, int* status, void* workspace, size_t workspace_bytes,
                    void* stream);

/* ---- training-time augmentation of a uint8 batch of line images (SURVEY.md 8(f) row 2) ----------------------
 * htrvt_augment_lines replaces the per-image PIL / OpenCV / scikit-image work of `SameTrCollate`
 * (model_v1/data/dataset.py:13-45): RandomTransform's projective warp + resize (model_v1/data/transform.py:164-230),
 * cv2 erode / dilate with an all-ones rectangle (transform.py:11-33) and torchvision ColorJitter's brightness /
 * contrast on grey images, one CTA per image, one launch per batch.  The random decisions are drawn on the host in the
 * reference's order (htr-vt_b200/augment.py::draw_collate_params) and passed as one 128-byte record per image:
 *   double m[9] (inverse projective map), double w0, w1 (anti-aliasing weights), int warp, rows, cols (shape of the
 *   intermediate warped image), gauss, jit_n, jit_op[2] (0 brightness, 1 contrast), float jit_f[2], int pad.
 * in uint8 [B, H, W] (stride_b bytes between images), out uint8 [B, H, W]; morph 0 none / 1 erode / 2 dilate, the same
 * k_rows x k_cols rectangle and iteration count for the whole batch.  2 * H * W <= 220 KB of shared memory. */
int htrvt_augment_lines(const void* in, long long stride_b, void* out, const void* recs, int B, int H, int W,
                        int morph, int k_rows, int k_cols, int iterations, void* stream);

/* Launch policy of the tensor-core GEMM family (all htrvt_gemm_*, htrvt_linear_wgrad, htrvt_conv_* entry points): with
 * programmatic dependent launch (default; HTRVT_PDL=0 in the environment disables it) a GEMM's prologue - barrier
 * initialisation, TMEM allocation, descriptor prefetch - runs under the tail of the launch in front of it on the same
 * stream; its first access to a tensor waits for that launch to complete.  Results do not depend on the setting.  There
 * is no counterpart in the reference (cuBLAS / cuDNN pick their own launch attributes).  Returns the previous setting. */
int htrvt_set_pdl(int on);

/* ---- tcgen05 tap-GEMM: nn.Linear / nn.Conv2d forward, input gradient, weight gradient ------------------
 * flags (epilogue, run by 8 warps and kept light): 1 bf16 out (else fp32), 2 +bias, 16 accumulate into out
 * (TMA reduce-add store), 32 column statistics (conv fwd), 128 ReLU.  Outputs leave through TMA stores.
 * htrvt_gemm_tn : Y = X W^T          nn.Linear fwd: attn.qkv / attn.proj (model_v1/model/HTR_VT.py:29,37),
 *                                    timm Mlp fc1 (+GELU) / fc2 (:76), head (:238)
 * htrvt_gemm_nn : dX = dY W          the same layers' input gradient (autograd of F.linear)
 * htrvt_linear_wgrad : dW (+)= dY^T X  the same layers' weight gradient, fp32, split-K workspace
 * Fused activation of timm Mlp (fc1 -> nn.GELU, erf form; model_v1/model/HTR_VT.py:76):
 *   gemm_tn flags 4096: out = gelu(X W^T + bias) (bf16); `pre` (nullable bf16 [M,N], row stride ldp, N % 256 == 0)
 *   additionally receives the DERIVATIVE gelu'(X W^T + bias) (train mode: two TMA stores per epilogue box; gelu and
 *   gelu' share one evaluation of Phi and exp);
 *   gemm_nn gelu_u (nullable, bf16 [M,N] contiguous): dX = (dY W) * gelu_u, gelu_u = that saved derivative - fc2's
 *   input gradient and the activation's backward in one kernel, one multiply per element in the epilogue. */
int htrvt_gemm_tn(const void* X, long long ldx, const void* W, long long ldw, int M, int N, int K, int flags,
                  const float* bias, void* out, long long ldo, float alpha, void* pre, long long ldp, void* stream);
int htrvt_gemm_nn(const void* dY, long long lddy, const void* W, long long ldw, int M, int N, int K, int flags,
                  void* out, long long ldo, float alpha, const void* gelu_u, float* colsum /*nullable: fp32 [N] +=
                  column sums of dX (with gelu_u): fc1's bias gradient*/, void* stream);
size_t htrvt_wgrad_workspace_bytes(int Cout, int Cin, int n_taps, int M_pixels);
int htrvt_linear_wgrad(const void* dY, long long lddy, const void* X, long long ldx, int M, int Nout, int Kin,
                       float* grad, int accumulate, void* workspace, size_t workspace_bytes, void* stream);
/* conv3x3 / 1x1 of BasicBlock and the downsample branch (model_v1/model/resnet18.py:4-7,23-39,56-63):
 * x NHWC bf16 [NB,H,W,Cin], w bf16 [Cout][ks*ks][Cin], stride (sh,sw), pad ks/2, bias-free.
 * stats_partial (optional): fp32 [htrvt_conv_fwd_stats_rows()][2][Cout] zero-initialised by the caller;
 * receives per-warp-quadrant column sum / sum of squares of the stored bf16 output (BatchNorm batch statistics). */
int htrvt_conv_fwd(const void* x, int NB, int H, int W, int Cin, const void* w, int Cout, int ks, int sh, int sw,
                   void* y, float* stats_partial, int flags, const float* bias, const void* res, void* stream);
int htrvt_conv_fwd_stats_rows(int NB, int H, int W, int ks, int sh, int sw);
/* Forward stem tensors (activations, raw conv outputs, forward weight copies) are IEEE fp16 in the engine: same 16
 * bits and tensor-core rate as bf16, 3 more mantissa bits - train-mode BatchNorm on bf16 tensors alone costs ~3e-2 on
 * the logits (DESIGN.md 4).  htrvt_conv_fwd takes the fp16 form with flags bit 1024.  Gradients (dy, dx) stay bf16
 * for their range, and because tcgen05 kind::f16 needs BOTH operands of an MMA in one format (a bf16 x fp16 descriptor
 * is an illegal instruction on B200) the backward GEMMs take bf16 only: the engine keeps bf16 copies of the
 * activations for the weight gradients (written by the same kernels that write the fp16 tensors) and bf16 transposed
 * weights for the input gradients. */
int htrvt_conv_dgrad(const void* dy, int NB, int H, int W, int Cin, const void* w, const void* w_t, int Cout, int ks,
                     int sh, int sw, void* dx, int accumulate, void* stream);
int htrvt_conv_wgrad(const void* dy, const void* dy_t, const void* x, int NB, int H, int W, int Cin, int Cout, int ks,
                     int sh, int sw, float* grad_oihw, int accumulate, void* workspace, size_t workspace_bytes,
                     void* stream);
/* split-K slices reduce-add (TMA) straight into grad_tapmajor fp32 [Cout][ks*ks][Cin] (+=): no partial sums, no
 * reduce kernel; htrvt_unpack_conv_grads then adds all tap-major gradients of a step into the OIHW parameters' .grad */
int htrvt_conv_wgrad_acc(const void* dy, const void* dy_t, const void* x, int NB, int H, int W, int Cin, int Cout,
                         int ks, int sh, int sw, float* grad_tapmajor, void* stream);
/* the same contraction transposed: grad_tco fp32 [ks*ks][Cin][Cout] (+=); rows of the GEMM = (tap, input channel),
 * columns = Cout: no padded MMA rows for Cout = 192 / 384 and CTA pairs for every shape (Cin % 64 == 0).
 * htrvt_unpack_conv_grads takes this layout with taps[i] = -(ks*ks). */
int htrvt_conv_wgrad_acc_t(const void* dy, const void* x, int NB, int H, int W, int Cin, int Cout, int ks, int sh,
                           int sw, float* grad_tco, void* stream);
/* 3x3, horizontal stride 1: two live accumulators share the dY tile and read x through two staged windows (the
 * three horizontal taps = one window at row offsets 0 / 1 / 2).  grad_atoms fp32 [3][Cin/64][3][64][Cout] (+=);
 * htrvt_unpack_conv_grads takes this layout with taps[i] = -1009. */
int htrvt_conv_wgrad_acc_w(const void* dy, const void* x, int NB, int H, int W, int Cin, int Cout, int sh,
                           float* grad_atoms, void* stream);
int htrvt_unpack_conv_grads(int n, const void* const* src_tapmajor, void* const* dst_oihw, const long long* numel,
                            const int* cin, const int* taps, void* stream);
/* bf16 [R][P][C] -> [R][C][P]: pixel-contiguous copy of a stem gradient (dy_t above; tcgen05 runs an MN-major A
 * operand ~1.4x slower than a K-major one, so the weight-gradient GEMM is fed dY^T) */
int htrvt_transpose_px(const void* in, void* out, long long R, int P, int C, void* stream);

/* ---- attention -------------------------------------------------------------------------------------------
 * Replaces Attention.forward's `q @ k^T * scale -> softmax -> @ v -> transpose/reshape`
 * (model_v1/model/HTR_VT.py:32-36) and its backward.  qkv bf16 token-major [B][T][3][H][128] (the QKV projection
 * output as htrvt_gemm_tn writes it: no reshape/permute copy), out bf16 [B][T][H*128], lse fp32 [B][H][T],
 * dqkv bf16 [B][T][3][H][128].  T <= 128. */
int htrvt_attention_fwd(const void* qkv, int B, int H, int T, int hd, float scale, void* out, float* lse,
                        void* stream);
int htrvt_attention_bwd(const void* qkv, const void* out, const void* dout, const float* lse, int B, int H, int T,
                        int hd, float scale, void* dqkv, void* stream);

/* ---- attention of the windowed variant (model_window/model/HTR_VT.py:33-62 Attention.forward with
 * relative_position_bias_table, :114-154 Block._attend: roll by -shift, 16-token windows, roll back), T <= 256.
 * table: fp32 [2*Prel-1][H] or NULL; window: 0 (global) or 16; shift: 0, or 8 with window 16 (any T <= 256: the
 * sequence is zero-padded to a multiple of 16, padded keys masked, padded query rows not stored);
 * drop_p / seed: attention dropout as a counter-based hash of (seed, b, h, query token, key token) - the backward
 * regenerates the mask; drop_p must lie in [0, 1) (NaN, negative or >= 1: HTRVT_ERR_SHAPE, nothing launched).
 * dtable (+=) is accumulated with fp32 atomics.  workspace: partial dQ for global T > 128. */
int htrvt_attention2_fwd(const void* qkv, int B, int H, int T, int hd, float scale, const float* table, int Prel,
                         int window, int shift, float drop_p, unsigned long long seed, void* out, float* lse,
                         void* stream);
size_t htrvt_attention2_bwd_workspace_bytes(int B, int H, int T, int window);
int htrvt_attention2_bwd(const void* qkv, const void* out, const void* dout, const float* lse, int B, int H, int T,
                         int hd, float scale, const float* table, int Prel, int window, int shift, float drop_p,
                         unsigned long long seed, void* dqkv, float* dtable, void* workspace, size_t workspace_bytes,
                         void* stream);

/* ---- LayerNorms, tokens, elementwise ---------------------------------------------------------------------
 * sample_ln : parameter-free LayerNorm over all non-batch dims, eps 1e-5 (model_v1/model/HTR_VT.py:134-136,
 *             used at :224 on the image and :239 on the logits slab)
 * row_ln    : nn.LayerNorm(D, eps=1e-6) with affine (:68,75,169), fp32 residual stream in, bf16 GEMM operand out;
 *             the residual update `x + attn(...)` / `x + mlp(...)` (Block.forward :80-83) is fused in as `addend`;
 *             backward accumulates into the fp32 residual gradient and into dgamma / dbeta
 * tokens    : `x * mask + (1 - mask) * mask_token` then `+ pos_embed` (:212-220, 229-231)
 * gelu_fwd/bwd : nn.GELU (erf form) of timm Mlp; colsum_bf16: bias gradients; cast / pack: bf16 operand
 *             copies of the fp32 master weights ([out,in] and OIHW -> [Cout][taps][Cin]). */
int htrvt_sample_ln_fwd(const float* x, void* y, int y_is_bf16, float* mean, float* rstd, int B, int N, float eps,
                        void* stream);
int htrvt_sample_ln_bwd(const float* dy, const float* y, const float* rstd, void* dx_bf16, int B, int N, int C,
                        int ld_out, void* stream);
int htrvt_row_ln_fwd(const float* x, const void* addend_bf16, float* x_out, const float* gamma, const float* beta,
                     void* y_bf16, float* mean, float* rstd, int M, int D, float eps, void* stream);
int htrvt_row_ln_bwd_ctas(int M);
int htrvt_row_ln_bwd(const void* dy_bf16, const float* x, const float* mean, const float* rstd, const float* gamma,
                     float* gx, int accumulate, float* dgamma, float* dbeta, float* partial, int M, int D,
                     void* stream);
int htrvt_tokens_fwd(const void* tok, const float* mask, const float* mask_token, const float* pos, float* x,
                     int B, int T, int D, int tok_f16, void* stream);
int htrvt_tokens_bwd(const float* gx, const float* mask, void* dtok_bf16, float* dmask_token, float* partial, int B,
                     int T, int D, void* stream);
int htrvt_gelu_fwd(const void* u, void* a, long long n, void* stream);
int htrvt_gelu_bwd(const void* da, const void* u, void* du, long long n, void* stream);
/* out = a * b (bf16, n % 8 == 0): the activation backward from the gelu'(u) the fused fc1 forward saved (`pre`). */
int htrvt_mul_bf16(const void* a, const void* b, void* out, long long n, void* stream);
int htrvt_colsum_rows(int M);
int htrvt_colsum_bf16(const void* a, long long ld, int M, int N, float* out, int accumulate, float* partial,
                      void* stream);
int htrvt_cast_bf16(const float* src, void* dst, long long n, void* stream);
/* dst bf16 [M,N] = bf16(src); colsum fp32 [N] += column sums of dst: the residual-stream gradient becomes fc2's /
 * proj's dY and their bias gradients in one pass (N % 8 == 0, N <= 2048) */
int htrvt_cast_colsum_bf16(const float* src, void* dst, float* colsum, int M, int N, void* stream);
/* in-place inverted dropout (+ per-sample DropPath scale dp[b], nullable) on bf16 x[n]; counter-based mask keyed by
 * (seed, site, element index): the same call on the gradient regenerates the mask.  Replaces nn.Dropout / timm
 * DropPath of model_window (model_window/model/HTR_VT.py:21-23, 100-110, 263-273) in train mode.  p must lie in
 * [0, 1) (NaN, negative or >= 1: HTRVT_ERR_SHAPE, nothing launched). */
int htrvt_dropout_bf16(void* x, long long n, long long per_sample, float p, unsigned long long seed, unsigned site,
                       const float* dp, void* stream);
int htrvt_pack_weights(int n, const void* const* src, void* const* dst, const long long* numel, const int* cin,
                       const int* taps, const void* const* scale, const int* f16, void* stream);
int htrvt_pack_conv_weight(const float* w_oihw, void* dst, int Cout, int Cin, int taps, void* stream);

/* ---- conv stem: first conv, BatchNorm, ReLU, max-pool ------------------------------------------------------
 * conv1     : nn.Conv2d(1, C, 3, stride (2,1), pad 1) (model_v1/model/resnet18.py:48), direct (K = 9), + statistics
 * bn_*      : nn.BatchNorm2d(eps=1e-5, momentum 0.1) train (batch stats, running-stat + counter update) / eval,
 *             ReLU and the residual add of BasicBlock.forward (resnet18.py:23-39), and their backward
 * pool_*    : nn.MaxPool2d(3, stride (2,1), pad 1) (resnet18.py:51,77,82) fused with BN + ReLU; idx = arg-max byte */
int htrvt_conv1_fwd_zdim(int B);
int htrvt_conv1_fwd(const float* x, const float* w, void* raw_bf16, float* partial, int B, int H, int W, int C,
                    void* stream);
int htrvt_bn_finalize(const float* partial, int R, double count, const float* gamma, const float* beta,
                      float* running_mean, float* running_var, long long* num_batches_tracked, float momentum,
                      float eps, int training, float* mean, float* rstd, float* scale, float* shift, int C,
                      void* stream);
int htrvt_bn_act_fwd(const void* raw, const float* scale, const float* shift, const void* res, const void* raw2,
                     const float* scale2, const float* shift2, void* y, void* y_bf16 /*nullable*/, void* relu_mask_bits,
                     long long P, int C, int relu, int f16, void* stream);
int htrvt_pool_fwd(const void* raw, const float* scale, const float* shift, void* out, void* idx, int B, int H,
                   int W, int C, int f16, void* stream);
int htrvt_pool_bwd(const void* gout, int gout_is_f32, const void* idx, const void* raw, const float* scale,
                   const float* shift, void* gin, int B, int H, int W, int C, int raw_f16, void* stream);
/* BatchNorm-backward reduction fused into the epilogue of the GEMM that produces the gradient (DESIGN.md 2):
 * htrvt_conv_dgrad_bn = htrvt_conv_dgrad of a 3x3 stride-1 conv whose epilogue masks the gradient with the ReLU bits of
 * the layer in front (dx = g') and accumulates sums[0][Cin] += sum g', sums[1][Cin] += sum g' xhat (zeroed by the
 * caller; [3][Cin] like htrvt_bn_bwd's `partial`); htrvt_bn_bwd_apply is htrvt_bn_bwd's second pass on such a pair.
 * htrvt_conv_dgrad_bn returns HTRVT_ERR_SHAPE (-1) for shapes its kernel does not serve: run the unfused pair then. */
int htrvt_conv_dgrad_bn(const void* dy, int NB, int H, int W, int Cin, const void* w_t, int Cout, void* dx,
                        const void* raw_f16, const void* relu_mask_bits, const float* mean, const float* rstd,
                        float* sums, void* stream);
int htrvt_bn_bwd_apply(const void* g_masked, const void* raw_a, const float* mean_a, const float* rstd_a,
                       const float* gamma_a, float* dgamma_a, float* dbeta_a, void* d_a, long long P, int C,
                       const float* sums, int raw_f16, void* stream);
int htrvt_bn_bwd_ctas(long long P);
int htrvt_bn_bwd(const void* g, const void* relu_mask_bits, const void* raw_a, const float* mean_a, const float* rstd_a,
                 const float* gamma_a, float* dgamma_a, float* dbeta_a, void* d_a, const void* raw_b,
                 const float* mean_b, const float* rstd_b, const float* gamma_b, float* dgamma_b, float* dbeta_b,
                 void* d_b, void* gz, long long P, int C, float* partial, float* coef, int raw_f16, void* stream);
/* ---- fused stem head: conv1 -> BatchNorm -> ReLU -> MaxPool without materialising the conv output -----------
 * Replaces model_v1/model/resnet18.py:74-77 (conv1, bn1, relu, maxpool) and their backward.  The conv has one
 * input channel and K = 9, so its output is recomputed from the fp32 image wherever it is needed:
 * htrvt_stem_head_moments: 3x3-patch moments of x (moments[54]: 9 sums + 45 upper-triangular products) and the
 *   exact per-channel (sum, sum of squares) of the conv output, stats[2][C] -> htrvt_bn_finalize (R = 1);
 * htrvt_stem_head_fwd: pooled activation bf16 [B,Ho,W,C] + 4-bit arg-max codes [B,Ho,W,C/2] (NULL in eval mode;
 *   code = kh*3+kw of torch's arg-max, 15 = ReLU inactive);
 * htrvt_stem_head_bwd: one pass over the pooled gradient g -> dgamma, dbeta (bn1) and dW (conv1, [C][9]), all +=. */
int htrvt_stem_head_moment_ctas(void);
int htrvt_stem_head_bwd_ctas(void);
int htrvt_stem_head_moments(const float* x, const float* w, float* partial, float* moments, float* stats, int B,
                            int H, int W, int C, void* stream);
/* htrvt_stem_head_fwd runs the convolution on the tensor pipe (stemhead_tc.cu: fp16 hi/lo split operands, the fp32
 * result to ~2^-21) when W % 64 == 0 and the output is 16-bit, on the FP32 pipe otherwise; htrvt_stem_head_set_mode(0)
 * forces the FP32-pipe kernel (tests), (1) restores the default; returns the previous mode. */
int htrvt_stem_head_set_mode(int mode);
int htrvt_stem_head_fwd(const float* x, const float* w, const float* scale, const float* shift, void* out,
                        void* out_bf16 /*nullable*/, void* code, int B, int H, int W, int C, int out_fmt, void* stream);
int htrvt_stem_head_bwd(const void* g, const void* code, const float* x, const float* w, const float* moments,
                        const float* gamma, const float* mean, const float* rstd, float* dgamma, float* dbeta,
                        float* dw, float* partial, int B, int H, int W, int C, void* stream);
int htrvt_conv1_wgrad_ctas(void);
int htrvt_conv1_wgrad(const void* dy_bf16, const float* x, float* grad, int accumulate, float* partial, int B,
                      int H, int W, int C, void* stream);

/* ---- multi-tensor optimizer passes around the hot path (SURVEY.md 8f rank 1) -------------------------------
 * Replace the per-parameter loops of SAM (model_v1/utils/sam.py:15-59), torch.optim.AdamW as configured at
 * model_v1/train.py:93 and ModelEma.update (model_v1/utils/utils.py:158-173).  Arrays of n DEVICE pointers to fp32
 * tensors live on the HOST (they travel as kernel parameters, <= 192 tensors per launch); numel[i] elements each.
 * norm2: device double, zeroed by the caller, receives sum |g|^2 (adaptive: |abs(p) g|^2). */
int htrvt_mt_sqnorm(int n, void* const* g, void* const* p, const long long* numel, int adaptive, double* norm2,
                    void* stream);
int htrvt_mt_sam_first(int n, void* const* p, void* const* g, void* const* old_p, const long long* numel,
                       const double* norm2, float rho, int adaptive, void* stream);
int htrvt_mt_adamw(int n, void* const* p, void* const* g, void* const* exp_avg, void* const* exp_avg_sq,
                   void* const* old_p, const long long* numel, float lr, float beta1, float beta2, float eps,
                   float weight_decay, int step, void* stream);
int htrvt_mt_ema(int n, void* const* ema, void* const* src, const long long* numel, float decay, void* stream);

/* ---- callers either side of the encoder (SURVEY.md 8f rows 2, 3) ----------------------------------------------
 * htrvt_line_prep_u8: the loader's `u8 / 255`, right padding with 1.0 (model_v1/data/dataset.py:13-45, 104-135) and the
 * model's whole-sample LayerNorm (model_v1/model/HTR_VT.py:134-136, 224) in one kernel on the uint8 line image.
 * img: uint8 [B, H, ld] (ld >= W, both multiples of 4; sample_stride in bytes); widths: int32 [B] valid columns or NULL;
 * y: fp32 [B, H, W]; mean / rstd: fp32 [B] or NULL.
 * htrvt_edit_distance: Levenshtein distance of n (prediction, ground-truth) int32 id sequences (editdistance.eval in
 * model_v1/valid.py:49-75); sequence p starts at x_off[p] if x_off else p * x_stride; max_b_len <= 4095. */
int htrvt_line_prep_u8(const void* img, long long sample_stride, int ld, const int* widths, int B, int H, int W,
                       float* y, float* mean, float* rstd, float eps, void* stream);
int htrvt_edit_distance(const int* a, const int* a_off, int a_stride, const int* a_len, const int* b, const int* b_off,
                        int b_stride, const int* b_len, int n, int max_b_len, int* out, void* stream);

/* ---- fp32-parity mode (eval forward; csrc/exact.cu) -------------------------------------------------------------
 * north_star: logits within 1e-4 of the fp32 reference and greedy-decode strings identical end to end.  Every tensor
 * between kernels is fp32; the dense contractions stay on the tcgen05 tap GEMM with SPLIT-bf16 operands
 * (x = h + m + l, three bf16 planes; six accumulating launches h.h' + h.m' + m.h' + m.m' + h.l' + l.h' into an fp32
 * output: htrvt_gemm_tn with EPI_ACCUM, htrvt_conv_fwd with flags 2048 | 16).  These entry points are the fp32
 * element-wise steps in between; `planes` = bf16 [3][n] (nullable where noted).
 * Reference lines: model_v1/model/HTR_VT.py:27-39 (attention), :68-83 (block), :134-136 / :224 / :236-239 (LayerNorms),
 * model_window/model/HTR_VT.py:33-62, 114-154 (the windowed variant's attention), model_v1/model/resnet18.py:23-39,73-84
 * (BatchNorm eval, ReLU, residual, max-pool), timm Mlp (erf GELU). */
int htrvt_split3(const float* src, void* planes_bf16, long long n, void* stream);
int htrvt_bn_act_f32(const float* raw, const float* scale, const float* shift, const float* res, const float* raw2,
                     const float* scale2, const float* shift2, float* y /*nullable*/, void* planes_bf16 /*nullable*/,
                     long long P, int C, int relu, void* stream);
int htrvt_maxpool_f32(const float* in, float* out, int B, int H, int W, int C, void* stream);
int htrvt_tokens_f32(const float* tok, const float* mask, const float* mask_token, const float* pos, float* x, int B,
                     int T, int D, void* stream);
int htrvt_row_ln_f32(const float* x, const float* addend /*nullable*/, float* x_out /*nullable*/, const float* gamma,
                     const float* beta, float* y /*nullable*/, void* planes_bf16 /*nullable*/, int M, int D, float eps,
                     void* stream);
int htrvt_gelu_split(const float* u, void* planes_bf16, long long n, void* stream);
int htrvt_attention_f32(const float* qkv /*[B,T,3,H,hd]*/, int B, int H, int T, int hd, float scale,
                        float* out /*[B,T,H*hd]*/, void* stream);
/* softmax(q k^T * scale + bias) v of the windowed variant (model_window/model/HTR_VT.py:33-62 Attention.forward with
 * relative_position_bias_table, :114-154 Block._attend) in fp32: the semantics of htrvt_attention2_fwd without dropout
 * or lse.  qkv fp32 [B][T][3][H][128] as the split GEMM writes it, out fp32 [B][T][H*128]; table fp32 [2*Prel-1][H] or
 * NULL.  Accepts exactly the shapes htrvt_attention2_fwd accepts (same HTRVT_ERR_SHAPE rules). */
int htrvt_attention2_f32(const float* qkv, int B, int H, int T, int hd, float scale, const float* table, int Prel,
                         int window, int shift, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HTRVT_H_ */
