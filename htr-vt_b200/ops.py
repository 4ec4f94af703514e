"""Thin torch-tensor -> C-ABI call layer (raw device pointers, current CUDA stream).

PyTorch is used here for device memory and streams only; all arithmetic runs in csrc/*.cu.
"""
import collections
import ctypes

import torch

from ._lib import HtrvtError, check, lib
from .wordlm import WordNGramLM

EPI_BF16, EPI_BIAS, _EPI_2, _EPI_3, EPI_ACCUM, EPI_STATS, _EPI_6, EPI_RELU = (1 << i for i in range(8))
EPI_F16 = 1 << 10
EPI_GELU = 1 << 12
# storage format of the FORWARD stem tensors (activations, raw conv outputs, forward conv-weight copies): IEEE fp16 -
# same 16 bits / tensor-core rate as bf16 with 3 more mantissa bits; gradients stay bf16 (DESIGN.md 4)
STEM_DTYPE = torch.float16


def _is_f16(t):
    return int(t is not None and t.dtype == torch.float16)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_raw_device = getattr(torch._C, "_cuda_getDevice", None)


def _stream():
    """Handle of torch's current stream on the current device.  Called once per kernel launch (~250 times per training
    step): the two raw C entry points cost ~0.3 us, `torch.cuda.current_stream().cuda_stream` ~15 us."""
    if _raw_stream is not None and _raw_device is not None:
        return ctypes.c_void_p(_raw_stream(_raw_device()))
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise HtrvtError("htr-vt_b200 kernels need CUDA tensors (there is no CPU fallback)")


def set_pdl(on) -> bool:
    """Programmatic dependent launch of the tap-GEMM family (htrvt_set_pdl); returns the previous setting."""
    return bool(lib().htrvt_set_pdl(int(bool(on))))


_ws_cache = {}


def workspace(nbytes: int, device) -> torch.Tensor:
    """Grow-only per-device scratch buffer (owned by PyTorch's caching allocator)."""
    key = (device.type, device.index)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf


# ------------------------------------------------------------------------------------------------
# GEMMs
# ------------------------------------------------------------------------------------------------
def gemm_tn(x, w, out, *, bias=None, relu=False, accumulate=False, flags=0, alpha=1.0, gelu=False, pre=None):
    """out[M,N] (+)= epilogue(alpha * x[M,K] @ w[N,K]^T).  x, w bf16 row-major; out bf16 or fp32 [M, N] view.
    gelu: out = gelu(... + bias) (erf form, bf16 out); pre (bf16 [M,N]): also receives gelu'(... + bias), the factor the
    backward multiplies by (gemm_nn's gelu_u / mul_bf16)."""
    _need_cuda(x, w, out)
    M, K = x.shape
    N = w.shape[0]
    f = flags | (EPI_BF16 if out.dtype == torch.bfloat16 else 0) | (EPI_BIAS if bias is not None else 0) \
        | (EPI_RELU if relu else 0) | (EPI_ACCUM if accumulate else 0) | (EPI_GELU if gelu else 0)
    check(lib().htrvt_gemm_tn(_p(x), x.stride(0), _p(w), w.stride(0), M, N, K, f, _p(bias), _p(out), out.stride(0),
                              alpha, _p(pre), pre.stride(0) if pre is not None else 0, _stream()), "htrvt_gemm_tn")
    return out


def gemm_nn(dy, w, out, *, accumulate=False, alpha=1.0, gelu_u=None, colsum=None):
    """out[M,N] (+)= dy[M,K] @ w[K,N]   (w row-major [K,N]: the nn.Linear weight itself for dgrad).
    gelu_u (bf16 [M,N] contiguous): out = (dy @ w) * gelu_u, gelu_u = the gelu' saved by gemm_tn(gelu=True, pre=...);
    colsum (fp32 [N], with gelu_u) += column sums of
    out (the bias gradient of the layer in front of the activation)."""
    _need_cuda(dy, w, out)
    M, K = dy.shape
    N = w.shape[1]
    f = (EPI_BF16 if out.dtype == torch.bfloat16 else 0) | (EPI_ACCUM if accumulate else 0)
    if gelu_u is not None and (not gelu_u.is_contiguous() or gelu_u.shape != out.shape or not out.is_contiguous()):
        raise HtrvtError("gemm_nn: gelu_u must be a contiguous bf16 [M, N] tensor like out")
    check(lib().htrvt_gemm_nn(_p(dy), dy.stride(0), _p(w), w.stride(0), M, N, K, f, _p(out), out.stride(0), alpha,
                              _p(gelu_u), _p(colsum), _stream()), "htrvt_gemm_nn")
    return out


def linear_wgrad(dy, x, grad, *, accumulate=True):
    """grad[N,K] (+)= dy[M,N]^T @ x[M,K]  (fp32 grad)."""
    _need_cuda(dy, x, grad)
    M, N = dy.shape
    K = x.shape[1]
    # split-K slices reduce-add straight into `grad`: the entry point takes no scratch (its workspace arguments are kept
    # for the ABI), so the call is safe on any stream
    check(lib().htrvt_linear_wgrad(_p(dy), dy.stride(0), _p(x), x.stride(0), M, N, K, _p(grad), int(accumulate),
                                   _p(None), 0, _stream()), "htrvt_linear_wgrad")
    return grad


def _need_bf16(*ts):
    for t in ts:
        if t is not None and t.dtype != torch.bfloat16:
            raise HtrvtError("backward GEMM operands must be bf16 (tcgen05 takes one 16-bit format per MMA; pass the "
                             "bf16 copy of a forward activation)")


def conv_wgrad_acc(dy, x, ks, sh, sw, grad_tapmajor):
    """grad_tapmajor fp32 [Cout, ks*ks, Cin] += dy^T x_shifted (split-K slices reduce-add in place, no reduce kernel)."""
    _need_cuda(dy, x, grad_tapmajor)
    _need_bf16(dy, x)
    N, H, W, Cin = x.shape
    Cout = dy.shape[-1]
    check(lib().htrvt_conv_wgrad_acc(_p(dy), _p(None), _p(x), N, H, W, Cin, Cout, ks, sh, sw, _p(grad_tapmajor),
                                     _stream()), "htrvt_conv_wgrad_acc")
    return grad_tapmajor


def conv_wgrad_acc_t(dy, x, ks, sh, sw, grad_tco):
    """grad_tco fp32 [ks*ks, Cin, Cout] += x_shifted^T dy (transposed weight-gradient GEMM, CTA pairs for every shape)."""
    _need_cuda(dy, x, grad_tco)
    _need_bf16(dy, x)
    N, H, W, Cin = x.shape
    Cout = dy.shape[-1]
    check(lib().htrvt_conv_wgrad_acc_t(_p(dy), _p(x), N, H, W, Cin, Cout, ks, sh, sw, _p(grad_tco), _stream()),
          "htrvt_conv_wgrad_acc_t")
    return grad_tco


def conv_wgrad_acc_w(dy, x, sh, grad_atoms):
    """3x3 conv, horizontal stride 1: grad_atoms fp32 [3, Cin/64, 3, 64, Cout] += (two-accumulator, window-sharing
    weight-gradient GEMM).  unpack_conv_grads(..., layout="atoms") permutes it into OIHW."""
    _need_cuda(dy, x, grad_atoms)
    _need_bf16(dy, x)
    N, H, W, Cin = x.shape
    Cout = dy.shape[-1]
    check(lib().htrvt_conv_wgrad_acc_w(_p(dy), _p(x), N, H, W, Cin, Cout, sh, _p(grad_atoms), _stream()),
          "htrvt_conv_wgrad_acc_w")
    return grad_atoms


def unpack_conv_grads(pairs, transposed=False, layout=None):
    """pairs: list of (src, dst fp32 OIHW): dst += permute(src), one launch for all.
    src fp32 [Cout, taps, Cin] (conv_wgrad_acc) or, transposed=True, [taps, Cin, Cout] (conv_wgrad_acc_t)."""
    n = len(pairs)
    if n == 0:
        return
    src = (ctypes.c_void_p * n)()
    dst = (ctypes.c_void_p * n)()
    numel = (ctypes.c_longlong * n)()
    cin = (ctypes.c_int * n)()
    taps = (ctypes.c_int * n)()
    for i, (a, b) in enumerate(pairs):
        src[i], dst[i], numel[i] = a.data_ptr(), b.data_ptr(), b.numel()
        if layout == "atoms":                       # [3, Cin/64, 3, 64, Cout]
            cin[i], taps[i] = a.shape[1] * 64, -1009
        elif transposed:
            cin[i], taps[i] = a.shape[1], -a.shape[0]
        else:
            cin[i], taps[i] = a.shape[2], a.shape[1]
    check(lib().htrvt_unpack_conv_grads(n, src, dst, numel, cin, taps, _stream()), "htrvt_unpack_conv_grads")


def conv_out_hw(H, W, ks, sh, sw):
    pad = ks // 2
    return (H + 2 * pad - ks) // sh + 1, (W + 2 * pad - ks) // sw + 1


def conv_fwd(x, w, ks, sh, sw, y=None, stats=None, relu=False, nostore=False, bias=None, res=None):
    """x [N,H,W,Cin] NHWC, w [Cout, ks*ks, Cin] -> y [N,Ho,Wo,Cout] (raw conv output); x, w, y (and res) share ONE
    16-bit format: fp16 (the engine's forward stem) or bf16.
    stats: optional fp32 [rows, 2, Cout] per-tile column sum / sum-of-squares partials.
    bias fp32 [Cout] / res like y: y = [relu](conv + bias + res) in the epilogue (eval-mode BatchNorm folding)."""
    _need_cuda(x, w)
    N, H, W, Cin = x.shape
    Cout = w.shape[0]
    Ho, Wo = conv_out_hw(H, W, ks, sh, sw)
    if y is None:
        y = torch.empty((N, Ho, Wo, Cout), dtype=x.dtype, device=x.device)
    if not (x.dtype == w.dtype == y.dtype and (res is None or res.dtype == x.dtype)):
        raise HtrvtError("conv_fwd: x, w, y and res must share one 16-bit format")
    check(lib().htrvt_conv_fwd(_p(x), N, H, W, Cin, _p(w), Cout, ks, sh, sw, _p(y), _p(stats),
                               (EPI_RELU if relu else 0) | (256 if nostore else 0) | (EPI_F16 if _is_f16(x) else 0),
                               _p(bias), _p(res), _stream()),
          "htrvt_conv_fwd")
    return y


def conv_stats_rows(N, H, W, ks, sh, sw):
    return lib().htrvt_conv_fwd_stats_rows(N, H, W, ks, sh, sw)


def conv_dgrad(dy, w, x_shape, ks, sh, sw, dx=None, accumulate=False, w_t=None):
    """dy, dx bf16; w bf16 [Cout, taps, Cin] (not read when w_t is given, so the forward pass's fp16 copy may be passed
    along with it); w_t (optional) bf16 [Cin, taps, Cout]: K-major B operand (CTA-pair kernel)."""
    _need_cuda(dy, w)
    N, H, W, Cin = x_shape
    Cout = w.shape[0]
    if dx is None:
        dx = torch.zeros(x_shape, dtype=torch.bfloat16, device=dy.device) if (ks == 1 and (sh > 1 or sw > 1)) \
            else torch.empty(x_shape, dtype=torch.bfloat16, device=dy.device)
    if dy.dtype != torch.bfloat16 or (w_t is None and w.dtype != torch.bfloat16) or \
            (w_t is not None and w_t.dtype != torch.bfloat16):
        raise HtrvtError("conv_dgrad operands must be bf16 (one 16-bit format per MMA; gradients are bf16)")
    check(lib().htrvt_conv_dgrad(_p(dy), N, H, W, Cin, _p(w), _p(w_t), Cout, ks, sh, sw, _p(dx), int(accumulate),
                                 _stream()),
          "htrvt_conv_dgrad")
    return dx


def transpose_px(dy):
    """dy bf16 [N,Ho,Wo,C] -> [N,Ho,C,Wo] (pixels contiguous): the K-major dY^T operand of conv_wgrad."""
    N, Ho, Wo, C = dy.shape
    out = torch.empty((N, Ho, C, Wo), dtype=torch.bfloat16, device=dy.device)
    check(lib().htrvt_transpose_px(_p(dy), _p(out), N * Ho, Wo, C, _stream()), "htrvt_transpose_px")
    return out


def conv_wgrad(dy, x, ks, sh, sw, grad_oihw, accumulate=True, transpose=False):
    _need_cuda(dy, x, grad_oihw)
    _need_bf16(dy, x)
    N, H, W, Cin = x.shape
    Cout = dy.shape[-1]
    Ho, Wo = conv_out_hw(H, W, ks, sh, sw)
    nbytes = lib().htrvt_wgrad_workspace_bytes(Cout, Cin, ks * ks, Wo)
    ws = workspace(nbytes, dy.device)
    # measured on B200: the K-major-A kernel is ~8 % faster than the pixel-major one, less than the separate
    # transpose costs, so the transposed operand is opt-in (worth it only if a producer writes dY^T for free)
    dy_t = transpose_px(dy) if (transpose and Wo % 8 == 0 and N * Ho <= 65535) else None
    check(lib().htrvt_conv_wgrad(_p(dy), _p(dy_t), _p(x), N, H, W, Cin, Cout, ks, sh, sw, _p(grad_oihw), int(accumulate),
                                 _p(ws), ws.numel(), _stream()), "htrvt_conv_wgrad")
    return grad_oihw


# ------------------------------------------------------------------------------------------------
# Attention
# ------------------------------------------------------------------------------------------------
def attention_fwd(qkv, out, lse, scale):
    """qkv bf16 [B,T,3,H,hd] (token-major projection output) -> out bf16 [B,T,H*hd]; lse fp32 [B,H,T]."""
    _need_cuda(qkv, out)
    B, T, _, H, hd = qkv.shape
    check(lib().htrvt_attention_fwd(_p(qkv), B, H, T, hd, scale, _p(out), _p(lse), _stream()), "htrvt_attention_fwd")
    return out


def attention_bwd(qkv, out, dout, lse, dqkv, scale):
    """-> dqkv bf16 [B,T,3,H,hd] (token-major gradient of the qkv projection output)."""
    _need_cuda(qkv, out, dout, lse, dqkv)
    B, T, _, H, hd = qkv.shape
    check(lib().htrvt_attention_bwd(_p(qkv), _p(out), _p(dout), _p(lse), B, H, T, hd, scale, _p(dqkv), _stream()),
          "htrvt_attention_bwd")
    return dqkv


def attention2_fwd(qkv, out, lse, scale, table=None, prel=0, window=0, shift=0, drop_p=0.0, seed=0):
    """Windowed-variant attention (T <= 256): relative-position bias table fp32 [2*prel-1, H] (None: no bias),
    window 0 (global) or 16 (16-token windows over the sequence rolled by -shift), attention dropout drop_p."""
    _need_cuda(qkv, out)
    B, T, _, H, hd = qkv.shape
    check(lib().htrvt_attention2_fwd(_p(qkv), B, H, T, hd, scale, _p(table), prel, window, shift, drop_p, seed, _p(out),
                                     _p(lse), _stream()), "htrvt_attention2_fwd")
    return out


def attention2_bwd(qkv, out, dout, lse, dqkv, scale, table=None, prel=0, window=0, shift=0, dtable=None, drop_p=0.0,
                   seed=0):
    """-> dqkv bf16 [B,T,3,H,hd]; dtable fp32 [2*prel-1, H] accumulated (+=) when given."""
    _need_cuda(qkv, out, dout, lse, dqkv)
    B, T, _, H, hd = qkv.shape
    nbytes = lib().htrvt_attention2_bwd_workspace_bytes(B, H, T, window)
    ws = workspace(nbytes, qkv.device) if nbytes else None
    check(lib().htrvt_attention2_bwd(_p(qkv), _p(out), _p(dout), _p(lse), B, H, T, hd, scale, _p(table), prel, window,
                                     shift, drop_p, seed, _p(dqkv), _p(dtable), _p(ws), ws.numel() if ws is not None else 0,
                                     _stream()), "htrvt_attention2_bwd")
    return dqkv


# ------------------------------------------------------------------------------------------------
# CTC + decode
# ------------------------------------------------------------------------------------------------
def ctc_loss_grad(x, targets, input_lengths, target_lengths, *, layout, is_logprob, want_grad=True,
                  max_target_len=-1, grad_scale=None, grad_scale_const=1.0):
    """x: fp32 logits [B,T,C] (layout 'btc') or log-probs [T,B,C] (layout 'tbc').
    Returns (nll [B] fp32, grad with the shape of x or None)."""
    _need_cuda(x)                      # lengths / targets may live on the host (valid.py:33 passes a CPU preds_size)
    if x.dtype != torch.float32 or x.stride(-1) != 1:
        raise HtrvtError("ctc_loss_grad expects fp32 input with a contiguous class axis")
    if layout == "btc":
        B, T, C = x.shape
        sb, st = x.stride(0), x.stride(1)
    else:
        T, B, C = x.shape
        sb, st = x.stride(1), x.stride(0)
    dev = x.device
    tg = targets.to(device=dev, dtype=torch.int32)
    tl = target_lengths.to(device=dev, dtype=torch.int32).contiguous()
    il = None if input_lengths is None else input_lengths.to(device=dev, dtype=torch.int32).contiguous()
    if tg.dim() == 2:
        tgt_stride = tg.stride(0)
        tg = tg.contiguous()
        tgt_stride = tg.stride(0)
    else:
        tg = tg.contiguous()
        tgt_stride = 0
    nll = torch.empty(B, dtype=torch.float32, device=dev)
    grad = torch.empty_like(x) if want_grad else None
    if grad is not None:
        gsb, gst = (grad.stride(0), grad.stride(1)) if layout == "btc" else (grad.stride(1), grad.stride(0))
    else:
        gsb = gst = 0
    nbytes = lib().htrvt_ctc_workspace_bytes(B, T, C, max_target_len)
    ws = workspace(nbytes, dev) if nbytes else None
    check(lib().htrvt_ctc_loss_grad(_p(x), sb, st, int(is_logprob), _p(tg), tgt_stride, _p(il), _p(tl), B, T, C,
                                    max_target_len, _p(nll), _p(grad), gsb, gst, _p(grad_scale), grad_scale_const,
                                    _p(ws), ws.numel() if ws is not None else 0, _stream()), "htrvt_ctc_loss_grad")
    return nll, grad


def greedy_decode_ids(logits, n_character, lengths=None, layout="btc", want_raw=False):
    """argmax + collapse on device.  Returns (ids [B,T] int32, lens [B] int32, raw [B,T] int32 | None)."""
    _need_cuda(logits)
    if logits.dtype != torch.float32 or logits.stride(-1) != 1:
        raise HtrvtError("greedy_decode expects fp32 logits with a contiguous class axis")
    if layout == "btc":
        B, T, C = logits.shape
        sb, st = logits.stride(0), logits.stride(1)
    else:
        T, B, C = logits.shape
        sb, st = logits.stride(1), logits.stride(0)
    dev = logits.device
    ids = torch.empty((B, T), dtype=torch.int32, device=dev)
    lens = torch.empty(B, dtype=torch.int32, device=dev)
    raw = torch.empty((B, T), dtype=torch.int32, device=dev) if want_raw else None
    ln = None if lengths is None else lengths.to(device=dev, dtype=torch.int32).contiguous()
    check(lib().htrvt_greedy_decode(_p(logits), sb, st, B, T, C, _p(ln), n_character, _p(ids), _p(lens), _p(raw),
                                    _stream()), "htrvt_greedy_decode")
    return ids, lens, raw


def _beam_io(name, log_probs, beam_size, lengths, layout, ctc_scores=False):
    """The common part of the beam decoders: checks the log-probs, -> (B, T, C, K, sb, st, lengths int32 | None, outs)
    with outs = [ids [B,K,T] int32, lens [B,K] int32, scores [B,K] float64 (, ctc_scores [B,K] float64)]."""
    _need_cuda(log_probs)
    if log_probs.dtype != torch.float32 or log_probs.stride(-1) != 1:
        raise HtrvtError("%s expects fp32 log-probs with a contiguous class axis" % name)
    if layout == "btc":
        B, T, C = log_probs.shape
        sb, st = log_probs.stride(0), log_probs.stride(1)
    else:
        T, B, C = log_probs.shape
        sb, st = log_probs.stride(1), log_probs.stride(0)
    dev = log_probs.device
    K = int(beam_size)
    outs = [torch.empty((B, K, T), dtype=torch.int32, device=dev), torch.empty((B, K), dtype=torch.int32, device=dev)]
    outs += [torch.empty((B, K), dtype=torch.float64, device=dev) for _ in range(2 if ctc_scores else 1)]
    ln = None if lengths is None else lengths.to(device=dev, dtype=torch.int32).contiguous()
    return B, T, C, K, sb, st, ln, outs


def ctc_kbest_paths(log_probs, beam_size, lengths=None, layout="tbc"):
    """K best alignment paths per line, collapsed (model_window/test_with_kenlm.py:25-51 on device).
    log_probs fp32 [T,B,C] ("tbc", the reference's layout) or [B,T,C] ("btc").
    Returns (ids [B,K,T] int32, lens [B,K] int32 (-1 = no such beam), scores [B,K] float64)."""
    B, T, C, K, sb, st, ln, outs = _beam_io("ctc_kbest_paths", log_probs, beam_size, lengths, layout)
    check(lib().htrvt_ctc_kbest_paths(_p(log_probs), sb, st, _p(ln), B, T, C, K, *map(_p, outs), _stream()),
          "htrvt_ctc_kbest_paths")
    return tuple(outs)


def ctc_prefix_beam(log_probs, beam_size, lengths=None, layout="tbc"):
    """CTC prefix beam search (csrc/prefix_beam.cu): the K most probable LABELLINGS per line, every beam entry carrying
    the summed probability of all its alignments - the search SURVEY.md 8(f) row 4 puts in place of the per-frame path
    beam of model_window/test_with_kenlm.py:25-59.  Same arguments and buffers as ctc_kbest_paths.
    Returns (ids [B,K,T] int32 zero padded, lens [B,K] int32 (-1 = no such prefix), scores [B,K] float64, best first)."""
    B, T, C, K, sb, st, ln, outs = _beam_io("ctc_prefix_beam", log_probs, beam_size, lengths, layout)
    check(lib().htrvt_ctc_prefix_beam(_p(log_probs), sb, st, _p(ln), B, T, C, K, *map(_p, outs), _stream()),
          "htrvt_ctc_prefix_beam")
    return tuple(outs)


def ctc_prefix_beam_lm(log_probs, beam_size, lm, alpha, beta=0.0, lengths=None, layout="tbc"):
    """ctc_prefix_beam with a character n-gram LM (lm.py::CharNGramLM) fused into the search: candidates rank by
    CTC log-prob + sum of (alpha * ln10 * log10 p(label | context) + beta), survivors by that plus the </s> term.
    Returns (ids [B,K,T] int32, lens [B,K] int32, scores [B,K] float64 (fused), ctc_scores [B,K] float64), in fused
    order.  alpha = beta = 0 reproduces ctc_prefix_beam's ids, lens and scores bit for bit."""
    if isinstance(lm, WordNGramLM):
        raise ValueError("a word LM scores the words of a lexicon: use ctc_prefix_beam_lex")
    B, T, C, K, sb, st, ln, outs = _beam_io("ctc_prefix_beam_lm", log_probs, beam_size, lengths, layout, True)
    if lm.table.device != log_probs.device:
        raise HtrvtError("ctc_prefix_beam_lm: the LM table lives on %s, the log-probs on %s"
                         % (lm.table.device, log_probs.device))
    check(lib().htrvt_ctc_prefix_beam_lm(_p(log_probs), sb, st, _p(ln), B, T, C, K, _p(lm.table), lm.slots, lm.order,
                                         _p(lm.token_map), lm.token_map.numel(), float(alpha), float(beta),
                                         *map(_p, outs), _stream()), "htrvt_ctc_prefix_beam_lm")
    return tuple(outs)


def ctc_prefix_beam_lex(log_probs, beam_size, lexicon, lm=None, alpha=0.0, beta=0.0, lengths=None, layout="tbc"):
    """ctc_prefix_beam (lm=None; alpha = beta = 0) or ctc_prefix_beam_lm (lm: a CharNGramLM) constrained to a word
    lexicon (lexicon.py::Lexicon): every maximal run of word characters in a returned labelling is a lexicon word.
    Ranking and scores are those of the unconstrained search; the lexicon only removes candidates.  lm may instead be
    a WordNGramLM built on this lexicon (wordlm.py): every finished word then adds alpha * ln10 * log10 p(word | <s>
    previous words) + beta, the line's end the </s> term, and a word being spelled ranks with its smear term.  Returns
    (ids [B,K,T] int32, lens [B,K] int32 (-1 = no such labelling; all K when the line has no accepted labelling),
    scores [B,K] float64 (fused; = ctc_scores without an LM), ctc_scores [B,K] float64)."""
    if isinstance(lm, WordNGramLM) and lm.lexicon is not lexicon:
        raise ValueError("ctc_prefix_beam_lex: the word LM was built on another lexicon")
    B, T, C, K, sb, st, ln, outs = _beam_io("ctc_prefix_beam_lex", log_probs, beam_size, lengths, layout, True)
    if lexicon.first.device != log_probs.device:
        raise HtrvtError("ctc_prefix_beam_lex: the lexicon lives on %s, the log-probs on %s"
                         % (lexicon.first.device, log_probs.device))
    if lm is not None and lm.table.device != log_probs.device:
        raise HtrvtError("ctc_prefix_beam_lex: the LM table lives on %s, the log-probs on %s"
                         % (lm.table.device, log_probs.device))
    lx = lexicon
    if isinstance(lm, WordNGramLM):
        check(lib().htrvt_ctc_prefix_beam_lex_wlm(_p(log_probs), sb, st, _p(ln), B, T, C, K, _p(lx.first),
                                                  _p(lx.label), _p(lx.child), _p(lx.word_end), lx.n_nodes,
                                                  _p(lx.is_word), lx.is_word.numel(), _p(lm.table), lm.slots, lm.order,
                                                  _p(lm.node_tok), _p(lm.smear), float(alpha), float(beta),
                                                  *map(_p, outs), _stream()), "htrvt_ctc_prefix_beam_lex_wlm")
        return tuple(outs)
    lm_args = ((None, 0, 0, None, 0) if lm is None else
               (lm.table, lm.slots, lm.order, lm.token_map, lm.token_map.numel()))
    check(lib().htrvt_ctc_prefix_beam_lex(_p(log_probs), sb, st, _p(ln), B, T, C, K, _p(lx.first), _p(lx.label),
                                          _p(lx.child), _p(lx.word_end), lx.n_nodes, _p(lx.is_word),
                                          lx.is_word.numel(), _p(lm_args[0]), lm_args[1], lm_args[2], _p(lm_args[3]),
                                          lm_args[4], float(alpha), float(beta), *map(_p, outs), _stream()),
          "htrvt_ctc_prefix_beam_lex")
    return tuple(outs)


CtcAlignment = collections.namedtuple("CtcAlignment", "path frame_scores spans token_scores score status")


def ctc_align(x, targets, target_lengths, input_lengths=None, layout="tbc", is_logprob=True):
    """Best CTC alignment of known labels per line (csrc/ctc_align.cu, blank = 0).
    x: fp32 log-probs (or raw logits with is_logprob=False) [T,B,C] ("tbc") or [B,T,C] ("btc"), class axis contiguous;
    targets int32 concatenated [sum L] or padded [B, Lpad]; lengths [B].  Lengths and targets may live on the host; the
    longest label is then the kernel's hint, else a device-side max is read back to size `spans`.
    Returns CtcAlignment of device tensors: path int32 [B,T] (-1 beyond a line's frames), frame_scores fp32 [B,T],
    spans int32 [B,Lmax,2] ([start, end) frames of each label), token_scores fp32 [B,Lmax], score float64 [B],
    status int32 [B] (0 aligned, 1 infeasible, 2 invalid line data)."""
    _need_cuda(x)
    if x.dtype != torch.float32 or x.stride(-1) != 1:
        raise HtrvtError("ctc_align expects fp32 input with a contiguous class axis")
    if layout == "btc":
        B, T, C = x.shape
        sb, st = x.stride(0), x.stride(1)
    elif layout == "tbc":
        T, B, C = x.shape
        sb, st = x.stride(1), x.stride(0)
    else:
        raise ValueError("layout must be 'tbc' or 'btc', got %r" % (layout,))
    dev = x.device
    if not torch.is_tensor(target_lengths):
        target_lengths = torch.as_tensor(target_lengths, dtype=torch.int32)
    if target_lengths.device.type == "cpu":
        hint = max(int(target_lengths.max()), 0) if target_lengths.numel() else 0
        lmax = hint
    else:
        hint = -1
        lmax = max(int(target_lengths.max()), 0) if target_lengths.numel() else 0
    tg = torch.as_tensor(targets).to(device=dev, dtype=torch.int32)
    tgt_stride = 0
    if tg.dim() == 2:
        tg = tg.contiguous()
        tgt_stride = tg.size(1)
    else:
        tg = tg.reshape(-1).contiguous()
    tl = target_lengths.to(device=dev, dtype=torch.int32).contiguous()
    il = None if input_lengths is None else torch.as_tensor(input_lengths).to(device=dev, dtype=torch.int32).contiguous()
    path = torch.empty((B, T), dtype=torch.int32, device=dev)
    frame_scores = torch.empty((B, T), dtype=torch.float32, device=dev)
    spans = torch.empty((B, lmax, 2), dtype=torch.int32, device=dev)
    token_scores = torch.empty((B, lmax), dtype=torch.float32, device=dev)
    score = torch.empty(B, dtype=torch.float64, device=dev)
    status = torch.empty(B, dtype=torch.int32, device=dev)
    nbytes = lib().htrvt_ctc_align_workspace_bytes(B, T, hint)
    ws = workspace(nbytes, dev) if nbytes else None
    check(lib().htrvt_ctc_align(_p(x), sb, st, int(bool(is_logprob)), _p(tg) if tg.numel() else None, tgt_stride,
                                _p(il), _p(tl), B, T, C, hint, _p(path), _p(frame_scores), _p(spans) if lmax else None,
                                lmax, _p(token_scores) if lmax else None, _p(score), _p(status), _p(ws),
                                ws.numel() if ws is not None else 0, _stream()), "htrvt_ctc_align")
    return CtcAlignment(path, frame_scores, spans, token_scores, score, status)


def augment_lines(img_u8, records, morph):
    """SameTrCollate's pixel work on a uint8 batch (csrc/augment.cu; model_v1/data/dataset.py:13-45).
    img_u8: CUDA uint8 [B, H, W] with contiguous rows; records: uint8 [B, 128] (CPU or CUDA; augment.py::pack_params);
    morph: (0 none | 1 erode | 2 dilate, k_rows, k_cols, iterations).  -> CUDA uint8 [B, H, W]."""
    _need_cuda(img_u8)
    if img_u8.dtype != torch.uint8 or img_u8.dim() != 3 or img_u8.stride(2) != 1 or img_u8.stride(1) != img_u8.shape[2]:
        raise HtrvtError("augment_lines expects uint8 [B, H, W] with contiguous images")
    B, H, W = img_u8.shape
    if records.dtype != torch.uint8 or tuple(records.shape) != (B, 128):
        raise HtrvtError("augment_lines expects one 128-byte record per image")
    rec = records.to(device=img_u8.device, non_blocking=True).contiguous()
    out = torch.empty((B, H, W), dtype=torch.uint8, device=img_u8.device)
    check(lib().htrvt_augment_lines(_p(img_u8), img_u8.stride(0), _p(out), _p(rec), B, H, W, int(morph[0]),
                                    int(morph[1]), int(morph[2]), int(morph[3]), _stream()), "htrvt_augment_lines")
    return out


def ctc_collapse(index_flat, lengths, n_character):
    """Collapse a sample-major index stream (reference decode() input).  -> (ids [B,Tmax], lens [B])."""
    _need_cuda(index_flat)
    dev = index_flat.device
    ln_host = lengths.detach().to("cpu", torch.int64)
    B = int(ln_host.numel())
    Tmax = int(ln_host.max()) if B else 0
    ln = ln_host.to(device=dev, dtype=torch.int32)
    offs = (torch.cumsum(ln_host, 0) - ln_host).to(device=dev, dtype=torch.int64)      # start of each line (one scan)
    idx = index_flat.contiguous()
    if idx.dtype not in (torch.int64, torch.int32):
        idx = idx.to(torch.int64)
    ids = torch.empty((B, max(Tmax, 1)), dtype=torch.int32, device=dev)
    lens = torch.empty(B, dtype=torch.int32, device=dev)
    check(lib().htrvt_ctc_collapse(_p(idx), int(idx.dtype == torch.int64), _p(ln), _p(offs), B, max(Tmax, 1),
                                   n_character, _p(ids), _p(lens), _stream()), "htrvt_ctc_collapse")
    return ids, lens


# ------------------------------------------------------------------------------------------------
# Normalisation / elementwise
# ------------------------------------------------------------------------------------------------
def _f32(n, dev):
    return torch.empty(n, dtype=torch.float32, device=dev)


def sample_ln_fwd(x, out_dtype, eps=1e-5):
    """x fp32 [B, ...] -> y (same shape, out_dtype), mean [B], rstd [B]."""
    _need_cuda(x)
    B = x.shape[0]
    N = x.numel() // B
    y = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    mean, rstd = _f32(B, x.device), _f32(B, x.device)
    check(lib().htrvt_sample_ln_fwd(_p(x), _p(y), int(out_dtype == torch.bfloat16), _p(mean), _p(rstd), B, N, eps,
                                    _stream()), "htrvt_sample_ln_fwd")
    return y, mean, rstd


def line_prep_u8(img, widths=None, eps=1e-5):
    """img uint8 [B, H, W] (rows may be strided) -> (y fp32 [B, H, W], mean [B], rstd [B]):
    u8 / 255, columns >= widths[b] read as 1.0, whole-sample LayerNorm - one kernel (SURVEY.md 8f row 2)."""
    _need_cuda(img)
    if img.dtype != torch.uint8 or img.dim() != 3 or img.stride(2) != 1:
        raise HtrvtError("line_prep_u8 expects uint8 [B, H, W] with contiguous rows")
    B, H, W = img.shape
    y = torch.empty((B, H, W), dtype=torch.float32, device=img.device)
    mean, rstd = _f32(B, img.device), _f32(B, img.device)
    wd = None if widths is None else widths.to(device=img.device, dtype=torch.int32).contiguous()
    check(lib().htrvt_line_prep_u8(_p(img), img.stride(0), img.stride(1), _p(wd), B, H, W, _p(y), _p(mean), _p(rstd),
                                   eps, _stream()), "htrvt_line_prep_u8")
    return y, mean, rstd


def edit_distance(a, a_len, b, b_len, a_off=None, b_off=None, max_b_len=None):
    """Levenshtein distance of n id-sequence pairs on device -> int32 [n].
    a / b: int32, either padded [n, stride] (x_off None) or concatenated 1-D with x_off int32 [n] start offsets."""
    _need_cuda(a, b)
    dev = a.device
    a = a.to(torch.int32).contiguous()
    b = b.to(device=dev, dtype=torch.int32).contiguous()
    a_len = a_len.to(device=dev, dtype=torch.int32).contiguous()
    b_len_d = b_len.to(device=dev, dtype=torch.int32).contiguous()
    n = a_len.numel()
    if max_b_len is None:
        max_b_len = b.shape[1] if (b_off is None and b.dim() == 2) else int(b_len.max()) if n else 0
    a_off = None if a_off is None else a_off.to(device=dev, dtype=torch.int32).contiguous()
    b_off = None if b_off is None else b_off.to(device=dev, dtype=torch.int32).contiguous()
    out = torch.empty(n, dtype=torch.int32, device=dev)
    check(lib().htrvt_edit_distance(_p(a), _p(a_off), a.stride(0) if a.dim() == 2 else 0, _p(a_len), _p(b), _p(b_off),
                                    b.stride(0) if b.dim() == 2 else 0, _p(b_len_d), n, int(max_b_len), _p(out),
                                    _stream()), "htrvt_edit_distance")
    return out


def sample_ln_bwd(dy, y, rstd, C, ld_out):
    """dy, y fp32 [B, T, C] -> dx bf16 [B*T, ld_out] (columns >= C zero)."""
    B = dy.shape[0]
    N = dy.numel() // B
    dx = torch.empty((B * (N // C), ld_out), dtype=torch.bfloat16, device=dy.device)
    check(lib().htrvt_sample_ln_bwd(_p(dy), _p(y), _p(rstd), _p(dx), B, N, C, ld_out, _stream()),
          "htrvt_sample_ln_bwd")
    return dx


def row_ln_fwd(x, gamma, beta, eps, addend=None):
    """y = LN(x [+ addend]) as bf16.  With `addend` (bf16 [M,D], the preceding GEMM's output) the residual update
    x_new = x + addend is fused here and returned (fp32).  -> (y, mean, rstd, x_new | x)"""
    M, D = x.shape
    y = torch.empty((M, D), dtype=torch.bfloat16, device=x.device)
    mean, rstd = _f32(M, x.device), _f32(M, x.device)
    x_new = torch.empty_like(x) if addend is not None else None
    check(lib().htrvt_row_ln_fwd(_p(x), _p(addend), _p(x_new), _p(gamma), _p(beta), _p(y), _p(mean), _p(rstd), M, D,
                                 eps, _stream()), "htrvt_row_ln_fwd")
    return y, mean, rstd, (x_new if addend is not None else x)


def row_ln_bwd(dy, x, mean, rstd, gamma, gx, accumulate, dgamma, dbeta):
    M, D = x.shape
    ctas = lib().htrvt_row_ln_bwd_ctas(M)
    partial = workspace(ctas * 2 * D * 4, x.device)
    check(lib().htrvt_row_ln_bwd(_p(dy), _p(x), _p(mean), _p(rstd), _p(gamma), _p(gx), int(accumulate), _p(dgamma),
                                 _p(dbeta), _p(partial), M, D, _stream()), "htrvt_row_ln_bwd")
    return gx


def tokens_fwd(tok, mask, mask_token, pos, B, T, D):
    x = torch.empty((B * T, D), dtype=torch.float32, device=tok.device)
    check(lib().htrvt_tokens_fwd(_p(tok), _p(mask), _p(mask_token if mask is not None else None), _p(pos), _p(x), B, T,
                                 D, _is_f16(tok), _stream()), "htrvt_tokens_fwd")
    return x


def tokens_bwd(gx, mask, dmask_token, B, T, D):
    dtok = torch.empty((B, T, D), dtype=torch.bfloat16, device=gx.device)
    partial = workspace(T * D * 4, gx.device)
    check(lib().htrvt_tokens_bwd(_p(gx), _p(mask), _p(dtok), _p(dmask_token if mask is not None else None),
                                 _p(partial), B, T, D, _stream()), "htrvt_tokens_bwd")
    return dtok


def gelu_fwd(u):
    a = torch.empty_like(u)
    check(lib().htrvt_gelu_fwd(_p(u), _p(a), u.numel(), _stream()), "htrvt_gelu_fwd")
    return a


def mul_bf16(a, b):
    """a * b (bf16): the activation backward from the saved gelu' when a dropout mask sits between activation and fc2."""
    out = torch.empty_like(a)
    check(lib().htrvt_mul_bf16(_p(a), _p(b), _p(out), a.numel(), _stream()), "htrvt_mul_bf16")
    return out


def gelu_bwd(da, u):
    du = torch.empty_like(u)
    check(lib().htrvt_gelu_bwd(_p(da), _p(u), _p(du), u.numel(), _stream()), "htrvt_gelu_bwd")
    return du


def dropout_(x, per_sample, p, seed, site, dp=None):
    """In-place inverted dropout of probability p (+ per-sample DropPath scale dp [B] fp32) on a bf16 tensor."""
    if p == 0.0 and dp is None:                  # (a p outside [0, 1) reaches the kernel entry, which refuses it)
        return x
    check(lib().htrvt_dropout_bf16(_p(x), x.numel(), per_sample, float(p), int(seed), int(site), _p(dp), _stream()),
          "htrvt_dropout_bf16")
    return x


def colsum_bf16(a, out, accumulate=True):
    M, N = a.shape
    rows = lib().htrvt_colsum_rows(M)
    partial = workspace(rows * N * 4, a.device)
    check(lib().htrvt_colsum_bf16(_p(a), a.stride(0), M, N, _p(out), int(accumulate), _p(partial), _stream()),
          "htrvt_colsum_bf16")
    return out


def cast_bf16(src, dst=None):
    if dst is None:
        dst = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device)
    check(lib().htrvt_cast_bf16(_p(src), _p(dst), src.numel(), _stream()), "htrvt_cast_bf16")
    return dst


def cast_colsum_bf16(src, colsum):
    """-> bf16 copy of src fp32 [M, N]; colsum fp32 [N] += its column sums (bias gradient of the layer whose dY it is)."""
    M, N = src.shape
    dst = torch.empty((M, N), dtype=torch.bfloat16, device=src.device)
    check(lib().htrvt_cast_colsum_bf16(_p(src), _p(dst), _p(colsum), M, N, _stream()), "htrvt_cast_colsum_bf16")
    return dst


def pack_conv_weight(w, dst=None):
    """fp32 OIHW -> bf16 [Cout, kh*kw, Cin]."""
    Cout, Cin, kh, kw = w.shape
    if dst is None:
        dst = torch.empty((Cout, kh * kw, Cin), dtype=torch.bfloat16, device=w.device)
    check(lib().htrvt_pack_conv_weight(_p(w), _p(dst), Cout, Cin, kh * kw, _stream()), "htrvt_pack_conv_weight")
    return dst


def pack_weights(items, pad_rows=None, names=None, conv_dtype=None, reuse=None):
    """items: list of (src fp32 tensor, kind[, scale]) with kind 'cast' ([out,in]), 'conv' (OIHW -> [Cout, taps, Cin];
    optional scale fp32 [Cout] folded in per output channel: eval-mode BatchNorm folding) or 'convT'.
    One launch for all of them.  pad_rows: {name: rows} allocates that 'cast' output with extra zero rows.
    Returns the list of 16-bit tensors: 'conv' copies in `conv_dtype` (default STEM_DTYPE = fp16, the forward stem's
    format), 'cast' and 'convT' (backward-only) copies in bf16.  reuse: the list a previous call with the same items
    returned - its tensors are overwritten instead of allocating ~50 new ones (the caller guarantees that nothing still
    reads them)."""
    conv_dtype = conv_dtype or STEM_DTYPE
    n = len(items)
    if reuse is not None and len(reuse) != n:
        reuse = None
    outs = []
    src = (ctypes.c_void_p * n)()
    dst = (ctypes.c_void_p * n)()
    numel = (ctypes.c_longlong * n)()
    cin = (ctypes.c_int * n)()
    taps = (ctypes.c_int * n)()
    scale = (ctypes.c_void_p * n)()
    f16 = (ctypes.c_int * n)()
    for i, item in enumerate(items):
        t, kind = item[0], item[1]
        scale[i] = item[2].data_ptr() if (len(item) > 2 and item[2] is not None) else None
        o = reuse[i] if reuse is not None else None
        if kind == "conv":
            Cout, Ci, kh, kw = t.shape
            if o is None:
                o = torch.empty((Cout, kh * kw, Ci), dtype=conv_dtype, device=t.device)
            cin[i], taps[i] = Ci, kh * kw
            f16[i] = int(conv_dtype == torch.float16)
        elif kind == "convT":                 # OIHW -> [Cin, taps, Cout] = plain transpose of [Cout, Cin*taps]
            Cout, Ci, kh, kw = t.shape
            if o is None:
                o = torch.empty((Ci, kh * kw, Cout), dtype=torch.bfloat16, device=t.device)
            cin[i], taps[i] = Cout, -1
        else:
            rows = pad_rows.get(names[i]) if (pad_rows and names) else None
            if o is None:
                if rows is not None and rows != t.shape[0]:      # (the pad rows are zero and stay zero: never written)
                    o = torch.zeros((rows, t.shape[1]), dtype=torch.bfloat16, device=t.device)
                else:
                    o = torch.empty(t.shape, dtype=torch.bfloat16, device=t.device)
            cin[i], taps[i] = 1, 0
        outs.append(o)
        src[i], dst[i], numel[i] = t.data_ptr(), o.data_ptr(), t.numel()
    check(lib().htrvt_pack_weights(n, src, dst, numel, cin, taps, scale, f16, _stream()), "htrvt_pack_weights")
    return outs


# ------------------------------------------------------------------------------------------------
# Stem
# ------------------------------------------------------------------------------------------------
def conv1_fwd(x, w, want_stats):
    """x fp32 [B,H,W]; w fp32 [C,1,3,3] -> raw bf16 [B,H/2,W,C], partial stats [R,2,C] | None."""
    B, H, W = x.shape
    C = w.shape[0]
    raw = torch.empty((B, H // 2, W, C), dtype=torch.bfloat16, device=x.device)
    R = min(B, 8) * (H // 2) * ((W + 127) // 128)
    partial = torch.empty((R, 2, C), dtype=torch.float32, device=x.device) if want_stats else None
    check(lib().htrvt_conv1_fwd(_p(x), _p(w), _p(raw), _p(partial), B, H, W, C, _stream()), "htrvt_conv1_fwd")
    return raw, partial


def bn_finalize(partial, count, gamma, beta, running_mean, running_var, nbt, training, momentum=0.1, eps=1e-5):
    """-> (mean, rstd, scale, shift) fp32 [C] each (one [4,C] buffer)."""
    C = gamma.numel()
    out = torch.empty((4, C), dtype=torch.float32, device=gamma.device)
    R = partial.shape[0] if partial is not None else 0
    check(lib().htrvt_bn_finalize(_p(partial), R, float(count), _p(gamma), _p(beta), _p(running_mean),
                                  _p(running_var), _p(nbt), momentum, eps, int(training), _p(out[0]), _p(out[1]),
                                  _p(out[2]), _p(out[3]), C, _stream()), "htrvt_bn_finalize")
    return out


def bn_act_fwd(raw, st, relu, res=None, raw2=None, st2=None, want_mask=False, want_bf16=False):
    """-> y, or (y, mask) with want_mask: mask uint8 [P, C/8] = ReLU mask bits consumed by bn_bwd.
    want_bf16 (train mode, fp16 forward tensors): also returns a bf16 copy of y as the LAST element - the operand of the
    next convolution's weight-gradient GEMM (which needs the format of dY); y itself when it already is bf16."""
    C = raw.shape[-1]
    P = raw.numel() // C
    y = torch.empty_like(raw)
    mask = torch.empty((P, C // 8), dtype=torch.uint8, device=raw.device) if want_mask else None
    y_bf = None
    if want_bf16:
        y_bf = y if raw.dtype == torch.bfloat16 else torch.empty(raw.shape, dtype=torch.bfloat16, device=raw.device)
    check(lib().htrvt_bn_act_fwd(_p(raw), _p(st[2]), _p(st[3]), _p(res), _p(raw2),
                                 _p(st2[2] if st2 is not None else None), _p(st2[3] if st2 is not None else None),
                                 _p(y), _p(y_bf if (y_bf is not None and y_bf is not y) else None), _p(mask), P, C,
                                 int(relu), _is_f16(raw), _stream()), "htrvt_bn_act_fwd")
    out = (y, mask) if want_mask else (y,)
    if want_bf16:
        out = out + (y_bf,)
    return out if len(out) > 1 else out[0]


def pool_fwd(raw, st, want_idx):
    B, H, W, C = raw.shape
    Ho = (H - 1) // 2 + 1
    out = torch.empty((B, Ho, W, C), dtype=raw.dtype, device=raw.device)
    idx = torch.empty((B, Ho, W, C), dtype=torch.uint8, device=raw.device) if want_idx else None
    check(lib().htrvt_pool_fwd(_p(raw), _p(st[2] if st is not None else None), _p(st[3] if st is not None else None),
                               _p(out), _p(idx), B, H, W, C, _is_f16(raw), _stream()), "htrvt_pool_fwd")
    return out, idx


def pool_bwd(gout, idx, in_shape, raw=None, st=None):
    B, H, W, C = in_shape
    gin = torch.empty(in_shape, dtype=torch.bfloat16, device=gout.device)
    check(lib().htrvt_pool_bwd(_p(gout), int(gout.dtype == torch.float32), _p(idx), _p(raw),
                               _p(st[2] if st is not None else None), _p(st[3] if st is not None else None), _p(gin),
                               B, H, W, C, _is_f16(raw), _stream()), "htrvt_pool_bwd")
    return gin


def bn_bwd(g, mask, raw_a, st_a, gamma_a, dgamma_a, dbeta_a, raw_b=None, st_b=None, gamma_b=None, dgamma_b=None,
           dbeta_b=None, want_gz=False, zero_sums=None):
    """-> (d_a, d_b | None, gz | None), all bf16 with the shape of raw_a.  g bf16; raw_a / raw_b in the forward
    stem's format (fp16, or bf16)."""
    C = raw_a.shape[-1]
    P = raw_a.numel() // C
    dev = raw_a.device
    d_a = torch.empty(raw_a.shape, dtype=torch.bfloat16, device=dev)
    d_b = torch.empty(raw_a.shape, dtype=torch.bfloat16, device=dev) if raw_b is not None else None
    gz = torch.empty(raw_a.shape, dtype=torch.bfloat16, device=dev) if want_gz else None
    if g.dtype != torch.bfloat16 or (raw_b is not None and raw_b.dtype != raw_a.dtype):
        raise HtrvtError("bn_bwd: gradient must be bf16, raw_a / raw_b one format")
    if zero_sums is None:                 # [3, C] fp32 zeros (engine: slices of one buffer cleared once per backward)
        zero_sums = torch.zeros(3 * C, dtype=torch.float32, device=dev)
    partial = zero_sums
    coef = None
    z = None
    check(lib().htrvt_bn_bwd(_p(g), _p(mask), _p(raw_a), _p(st_a[0]), _p(st_a[1]), _p(gamma_a), _p(dgamma_a),
                             _p(dbeta_a), _p(d_a), _p(raw_b), _p(st_b[0] if st_b is not None else z),
                             _p(st_b[1] if st_b is not None else z), _p(gamma_b), _p(dgamma_b), _p(dbeta_b), _p(d_b),
                             _p(gz), P, C, _p(partial), _p(coef), _is_f16(raw_a), _stream()), "htrvt_bn_bwd")
    return d_a, d_b, gz


def conv_dgrad_bn(dy, w_t, x_shape, raw, mask, st, sums):
    """Input gradient of a 3x3 stride-1 conv fused with the reduction pass of the BatchNorm backward of the layer in
    front: -> g' = (conv_transpose(dy, w)) * relu_mask as bf16 with the shape of `raw`, sums[0] += sum g',
    sums[1] += sum g' xhat (sums: fp32 [3*C] zeros).  Returns None when the fused kernel does not serve the shape."""
    _need_cuda(dy, w_t, raw)
    N, H, W, Cin = x_shape
    Cout = dy.shape[-1]
    if dy.dtype != torch.bfloat16 or w_t.dtype != torch.bfloat16 or raw.dtype != torch.float16 or mask is None:
        return None
    dx = torch.empty(x_shape, dtype=torch.bfloat16, device=dy.device)
    r = lib().htrvt_conv_dgrad_bn(_p(dy), N, H, W, Cin, _p(w_t), Cout, _p(dx), _p(raw), _p(mask), _p(st[0]), _p(st[1]),
                                  _p(sums), _stream())
    if r == -1:
        return None
    check(r, "htrvt_conv_dgrad_bn")
    return dx


def bn_bwd_apply(g_masked, raw_a, st_a, gamma_a, dgamma_a, dbeta_a, sums):
    """Second pass of bn_bwd on a masked gradient whose [3, C] sums already exist (conv_dgrad_bn) -> d_a bf16."""
    C = raw_a.shape[-1]
    P = raw_a.numel() // C
    d_a = torch.empty(raw_a.shape, dtype=torch.bfloat16, device=raw_a.device)
    check(lib().htrvt_bn_bwd_apply(_p(g_masked), _p(raw_a), _p(st_a[0]), _p(st_a[1]), _p(gamma_a), _p(dgamma_a),
                                   _p(dbeta_a), _p(d_a), P, C, _p(sums), _is_f16(raw_a), _stream()),
          "htrvt_bn_bwd_apply")
    return d_a


def stem_head_moments(x, w):
    """x fp32 [B,H,W], w fp32 [C,1,3,3] -> (moments fp32 [54], stats fp32 [1,2,C]): 3x3-patch moments of the image and
    the exact per-channel sum / sum of squares of the (never materialised) conv1 output."""
    _need_cuda(x, w)
    B, H, W = x.shape
    C = w.shape[0]
    moments = torch.empty(54, dtype=torch.float32, device=x.device)
    stats = torch.empty((1, 2, C), dtype=torch.float32, device=x.device)
    partial = workspace(lib().htrvt_stem_head_moment_ctas() * 54 * 4, x.device)
    check(lib().htrvt_stem_head_moments(_p(x), _p(w), _p(partial), _p(moments), _p(stats), B, H, W, C, _stream()),
          "htrvt_stem_head_moments")
    return moments, stats


def stem_head_fwd(x, w, st, want_code, out_dtype=None, want_bf16=False):
    """conv1 -> BN(scale/shift of st) -> ReLU -> MaxPool(3,(2,1),1).  -> (out [B,Ho,W,C] in STEM_DTYPE (fp16) unless
    out_dtype says otherwise, code uint8 | None[, bf16 copy of out with want_bf16: weight-gradient operand])."""
    _need_cuda(x, w)
    B, H, W = x.shape
    C = w.shape[0]
    Ho = (H // 2 - 1) // 2 + 1
    out = torch.empty((B, Ho, W, C), dtype=out_dtype or STEM_DTYPE, device=x.device)
    code = torch.empty((B, Ho, W, C // 2), dtype=torch.uint8, device=x.device) if want_code else None
    fmt = {torch.bfloat16: 0, torch.float16: 1, torch.float32: 2}[out.dtype]
    out_bf = None
    if want_bf16:
        out_bf = out if out.dtype == torch.bfloat16 else torch.empty(out.shape, dtype=torch.bfloat16, device=x.device)
    check(lib().htrvt_stem_head_fwd(_p(x), _p(w), _p(st[2]), _p(st[3]), _p(out),
                                    _p(out_bf if (out_bf is not None and out_bf is not out) else None), _p(code), B, H, W,
                                    C, fmt, _stream()), "htrvt_stem_head_fwd")
    return (out, code, out_bf) if want_bf16 else (out, code)


def stem_head_bwd(g, code, x, w, moments, gamma, st, dgamma, dbeta, dw):
    """One pass over the pooled gradient g bf16 [B,Ho,W,C]: dgamma, dbeta, dw (fp32, +=)."""
    _need_cuda(g, code, x)
    B, H, W = x.shape
    C = w.shape[0]
    if not g.is_contiguous():
        g = g.contiguous()
    partial = workspace(lib().htrvt_stem_head_bwd_ctas() * 11 * C * 4, x.device)
    check(lib().htrvt_stem_head_bwd(_p(g), _p(code), _p(x), _p(w), _p(moments), _p(gamma), _p(st[0]), _p(st[1]),
                                    _p(dgamma), _p(dbeta), _p(dw), _p(partial), B, H, W, C, _stream()),
          "htrvt_stem_head_bwd")


def conv1_wgrad(dy, x, grad, accumulate=True):
    B, H, W = x.shape
    C = dy.shape[-1]
    ctas = lib().htrvt_conv1_wgrad_ctas()
    partial = workspace(ctas * 9 * C * 4, x.device)
    check(lib().htrvt_conv1_wgrad(_p(dy), _p(x), _p(grad), int(accumulate), _p(partial), B, H, W, C, _stream()),
          "htrvt_conv1_wgrad")
    return grad


# ------------------------------------------------------------------------------------------------
# fp32-parity mode (csrc/exact.cu): split-bf16 operands on the tensor pipe, fp32 everywhere else
# ------------------------------------------------------------------------------------------------
# (activation plane, weight plane) products kept, smallest first so the fp32 output accumulates upwards;
# dropped: m.l', l.m', l.l' (<= 2^-24 relative)
SPLIT_TERMS = ((2, 0), (0, 2), (1, 1), (1, 0), (0, 1), (0, 0))


def split3(src):
    """fp32 tensor -> bf16 planes [3, *shape] with h + m + l == src to 24 bits."""
    _need_cuda(src)
    src = src.contiguous()
    planes = torch.empty((3,) + tuple(src.shape), dtype=torch.bfloat16, device=src.device)
    check(lib().htrvt_split3(_p(src), _p(planes), src.numel(), _stream()), "htrvt_split3")
    return planes


def gemm_tn_split(xp, wp, out, bias=None):
    """out fp32 [M,N] = x @ w^T (+ bias) from bf16 planes xp [3,M,K], wp [3,N,K]: six accumulating tcgen05 GEMMs."""
    for n, (i, j) in enumerate(SPLIT_TERMS):
        gemm_tn(xp[i], wp[j], out, accumulate=n > 0, bias=bias if n == len(SPLIT_TERMS) - 1 else None)
    return out


def conv_fwd_split(xp, wp, ks, sh, sw):
    """fp32 raw conv output [N,Ho,Wo,Cout] from bf16 planes xp [3,N,H,W,Cin], wp [3,Cout,ks*ks,Cin]."""
    _, N, H, W, Cin = xp.shape
    Cout = wp.shape[1]
    Ho, Wo = conv_out_hw(H, W, ks, sh, sw)
    y = torch.empty((N, Ho, Wo, Cout), dtype=torch.float32, device=xp.device)
    for n, (i, j) in enumerate(SPLIT_TERMS):
        check(lib().htrvt_conv_fwd(_p(xp[i]), N, H, W, Cin, _p(wp[j]), Cout, ks, sh, sw, _p(y), _p(None),
                                   2048 | (EPI_ACCUM if n > 0 else 0), _p(None), _p(None), _stream()),
              "htrvt_conv_fwd (fp32 output)")
    return y


def bn_act_f32(raw, st, relu, res=None, raw2=None, st2=None, want_y=True, want_planes=True):
    """fp32 BatchNorm(eval coefficients st[2], st[3]) + residual / second BN + ReLU -> (y fp32 | None, planes | None)."""
    C = raw.shape[-1]
    P = raw.numel() // C
    y = torch.empty_like(raw) if want_y else None
    planes = torch.empty((3,) + tuple(raw.shape), dtype=torch.bfloat16, device=raw.device) if want_planes else None
    check(lib().htrvt_bn_act_f32(_p(raw), _p(st[2]), _p(st[3]), _p(res), _p(raw2),
                                 _p(st2[2] if st2 is not None else None), _p(st2[3] if st2 is not None else None),
                                 _p(y), _p(planes), P, C, int(relu), _stream()), "htrvt_bn_act_f32")
    return y, planes


def maxpool_f32(x):
    B, H, W, C = x.shape
    out = torch.empty((B, (H - 1) // 2 + 1, W, C), dtype=torch.float32, device=x.device)
    check(lib().htrvt_maxpool_f32(_p(x), _p(out), B, H, W, C, _stream()), "htrvt_maxpool_f32")
    return out


def tokens_f32(tok, mask, mask_token, pos, B, T, D):
    x = torch.empty((B * T, D), dtype=torch.float32, device=tok.device)
    check(lib().htrvt_tokens_f32(_p(tok), _p(mask), _p(mask_token if mask is not None else None), _p(pos), _p(x), B, T,
                                 D, _stream()), "htrvt_tokens_f32")
    return x


def row_ln_f32(x, gamma, beta, eps, addend=None):
    """-> (planes bf16 [3,M,D] of LN(x + addend), x + addend fp32)."""
    M, D = x.shape
    planes = torch.empty((3, M, D), dtype=torch.bfloat16, device=x.device)
    x_new = torch.empty_like(x) if addend is not None else None
    check(lib().htrvt_row_ln_f32(_p(x), _p(addend), _p(x_new), _p(gamma), _p(beta), _p(None), _p(planes), M, D, eps,
                                 _stream()), "htrvt_row_ln_f32")
    return planes, (x_new if addend is not None else x)


def gelu_split(u):
    planes = torch.empty((3,) + tuple(u.shape), dtype=torch.bfloat16, device=u.device)
    check(lib().htrvt_gelu_split(_p(u), _p(planes), u.numel(), _stream()), "htrvt_gelu_split")
    return planes


def attention_f32(qkv, B, H, T, hd, scale):
    out = torch.empty((B * T, H * hd), dtype=torch.float32, device=qkv.device)
    check(lib().htrvt_attention_f32(_p(qkv), B, H, T, hd, scale, _p(out), _stream()), "htrvt_attention_f32")
    return out


def attention2_f32(qkv, B, H, T, hd, scale, table=None, prel=0, window=0, shift=0, out=None):
    """Windowed-variant attention in fp32 (eval: no dropout): qkv fp32 [B*T, 3*H*hd] -> fp32 [B*T, H*hd] (written
    into `out` when given).  Relative-position bias table fp32 [2*prel-1, H] (None: no bias), window 0 (global) or 16
    with shift 0 or 8, as attention2_fwd."""
    _need_cuda(qkv, table, out)
    if qkv.dtype != torch.float32 or not qkv.is_contiguous() or (table is not None and table.dtype != torch.float32):
        raise HtrvtError("attention2_f32 needs contiguous fp32 qkv and an fp32 bias table")
    if out is None:
        out = torch.empty((B * T, H * hd), dtype=torch.float32, device=qkv.device)
    elif out.dtype != torch.float32 or not out.is_contiguous() or out.numel() != B * T * H * hd:
        raise HtrvtError("attention2_f32: out must be a contiguous fp32 tensor of B*T*H*hd elements")
    check(lib().htrvt_attention2_f32(_p(qkv), B, H, T, hd, scale, _p(table), prel, window, shift, _p(out), _stream()),
          "htrvt_attention2_f32")
    return out


def launch_count() -> int:
    """Kernels launched by the library so far (host-side counter in the C library)."""
    fn = lib().htrvt_launch_count
    fn.restype = ctypes.c_ulonglong
    return int(fn())


# ------------------------------------------------------------------------------------------------
# Optional per-op CUDA-event profile (bench.py's roofline leg, tools/): PROFILE = [] enables it.
# ------------------------------------------------------------------------------------------------
PROFILE = None
# bumped by every kernel that rewrites parameters through raw pointers (SAM / AdamW / EMA): autograd's version counters
# do not see those writes, and the engine keys its eval-mode cache of packed bf16 weights on (versions, this epoch)
WEIGHT_EPOCH = 0


def weights_changed():
    global WEIGHT_EPOCH
    WEIGHT_EPOCH += 1


def _flops(name, a, kw):
    try:
        if name == "gemm_tn":
            return 2.0 * a[0].shape[0] * a[0].shape[1] * a[1].shape[0]
        if name == "gemm_nn":
            return 2.0 * a[0].shape[0] * a[0].shape[1] * a[1].shape[1]
        if name == "linear_wgrad":
            return 2.0 * a[0].shape[0] * a[0].shape[1] * a[1].shape[1]
        if name == "conv_fwd":
            x, w, ks, sh, sw = a[:5]
            Ho, Wo = conv_out_hw(x.shape[1], x.shape[2], ks, sh, sw)
            return 2.0 * x.shape[0] * Ho * Wo * w.shape[0] * ks * ks * x.shape[3]
        if name == "conv_dgrad":
            dy, w, xs, ks = a[:4]
            return 2.0 * dy.shape[0] * dy.shape[1] * dy.shape[2] * dy.shape[3] * ks * ks * xs[3]
        if name == "conv_dgrad_bn":
            dy, w_t, xs = a[:3]
            return 2.0 * dy.shape[0] * dy.shape[1] * dy.shape[2] * dy.shape[3] * 9 * xs[3]
        if name == "conv_wgrad_acc_w":
            dy, x = a[:2]
            return 2.0 * dy.shape[0] * dy.shape[1] * dy.shape[2] * dy.shape[3] * 9 * x.shape[3]
        if name in ("conv_wgrad_acc", "conv_wgrad_acc_t"):
            dy, x, ks = a[:3]
            return 2.0 * dy.shape[0] * dy.shape[1] * dy.shape[2] * dy.shape[3] * ks * ks * x.shape[3]
        if name == "conv_wgrad":
            dy, x, ks = a[:3]
            return 2.0 * dy.shape[0] * dy.shape[1] * dy.shape[2] * dy.shape[3] * ks * ks * x.shape[3]
        if name == "attention2_fwd":
            B, T, _, H, hd = a[0].shape
            return 4.0 * B * H * T * T * hd
        if name == "attention2_bwd":
            B, T, _, H, hd = a[0].shape
            return 10.0 * B * H * T * T * hd
        if name == "attention_fwd":
            B, T, _, H, hd = a[0].shape
            return 4.0 * B * H * T * T * hd
        if name == "attention_bwd":
            B, T, _, H, hd = a[0].shape
            return 10.0 * B * H * T * T * hd
        if name == "conv_fwd_split":                             # six bf16 products
            xp, wp, ks, sh, sw = a[:5]
            Ho, Wo = conv_out_hw(xp.shape[2], xp.shape[3], ks, sh, sw)
            return 6 * 2.0 * xp.shape[1] * Ho * Wo * wp.shape[1] * ks * ks * xp.shape[4]
        if name == "attention_f32":
            B, H, T, hd = a[1:5]
            return 4.0 * B * H * T * T * hd
        if name == "attention2_f32":
            B, H, T, hd = a[1:5]
            window = a[8] if len(a) > 8 else kw.get("window", 0)
            if window:                                           # every query sees the 16 keys of its window
                return 4.0 * B * H * ((T + window - 1) // window * window) * window * hd
            return 4.0 * B * H * T * T * hd
    except Exception:
        pass
    return 0.0


def _instrument():
    import functools
    g = globals()
    names = ["gemm_tn", "gemm_nn", "linear_wgrad", "conv_fwd", "conv_dgrad", "conv_dgrad_bn", "conv_wgrad", "conv_wgrad_acc", "conv_wgrad_acc_t", "conv_wgrad_acc_w", "unpack_conv_grads", "attention_fwd",
             "attention_bwd", "attention2_fwd", "attention2_bwd", "attention_f32", "attention2_f32", "split3", "conv_fwd_split", "bn_act_f32", "maxpool_f32", "tokens_f32", "row_ln_f32", "gelu_split", "ctc_loss_grad", "greedy_decode_ids", "ctc_collapse", "ctc_kbest_paths", "ctc_prefix_beam", "ctc_prefix_beam_lm", "ctc_prefix_beam_lex", "ctc_align", "augment_lines", "sample_ln_fwd", "sample_ln_bwd", "line_prep_u8", "edit_distance",
             "row_ln_fwd", "row_ln_bwd", "tokens_fwd", "tokens_bwd", "gelu_fwd", "gelu_bwd", "colsum_bf16", "cast_bf16", "cast_colsum_bf16", "dropout_",
             "pack_conv_weight", "pack_weights", "conv1_fwd", "bn_finalize", "bn_act_fwd", "pool_fwd", "pool_bwd", "bn_bwd", "bn_bwd_apply",
             "conv1_wgrad", "stem_head_moments", "stem_head_fwd", "stem_head_bwd"]
    for name in names:
        fn = g[name]

        def make(fn=fn, name=name):
            @functools.wraps(fn)
            def wrapper(*a, **kw):
                if PROFILE is None:
                    return fn(*a, **kw)
                e0 = torch.cuda.Event(enable_timing=True)
                e1 = torch.cuda.Event(enable_timing=True)
                e0.record()
                r = fn(*a, **kw)
                e1.record()
                PROFILE.append((name, _flops(name, a, kw), e0, e1))
                return r
            return wrapper
        g[name] = make()


_instrument()
