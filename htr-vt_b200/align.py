"""CTC forced alignment: where each character of a known transcription lies in the line.

ctc_align      the kernel's full output (path, frame and token scores, label spans, Viterbi score, status) for a batch;
forced_align   torchaudio.functional.forced_align's contract ([B, T, C] log-probs, padded targets) for any batch size;
align_text     strings in, character boxes in image pixels out, from the model's raw logits.
All three run csrc/ctc_align.cu (blank = 0); only the final per-line lists of align_text are built on the host.
"""
import torch

from . import ops
from ._lib import HtrvtError
from .ops import ctc_align  # noqa: F401  (public form)


def _lines(mask):
    return [int(i) for i in torch.nonzero(mask).reshape(-1).tolist()]


def forced_align(log_probs, targets, input_lengths=None, target_lengths=None, blank=0):
    """torchaudio.functional.forced_align for a batch: log_probs fp32 [B, T, C] (CUDA), targets [B, L] padded,
    input_lengths / target_lengths [B] (default: T and L for every line).  Returns (alignments int32 [B, T], scores
    fp32 [B, T]) on the device: the class of every frame and its log-prob; frames beyond a line's length hold -1 and 0.
    On exact ties the path is a true maximum (first of stay / previous / skip), where torchaudio can return a path
    below it.  Raises ValueError for blank != 0 or invalid label ids or lengths, HtrvtError (a RuntimeError, as
    torchaudio raises) naming the lines whose transcription cannot fit their frames."""
    if blank != 0:
        raise ValueError("forced_align implements blank = 0 (the library's convention), got blank=%d" % blank)
    if log_probs.dim() != 3:
        raise ValueError("log_probs must be [B, T, C], got shape %s" % (tuple(log_probs.shape),))
    targets = torch.as_tensor(targets)
    if targets.dim() != 2 or targets.size(0) != log_probs.size(0):
        raise ValueError("targets must be padded [B, L] with B = %d, got shape %s"
                         % (log_probs.size(0), tuple(targets.shape)))
    if target_lengths is None:
        target_lengths = torch.full((targets.size(0),), targets.size(1), dtype=torch.int32)
    r = ops.ctc_align(log_probs, targets, target_lengths, input_lengths, layout="btc", is_logprob=True)
    status = r.status.cpu()
    if bool((status == 2).any()):
        raise ValueError("forced_align: invalid label ids or lengths in lines %s" % _lines(status == 2))
    if bool((status == 1).any()):
        raise HtrvtError("forced_align: the targets of lines %s are too long for their input lengths"
                         % _lines(status == 1))
    return r.path, r.frame_scores


def align_text(logits, converter, texts, lengths=None, *, image_width=None, px_per_frame=None):
    """Character boxes of known line transcriptions.  logits: the model's fp32 output [B, T, C] (raw, no log-softmax);
    converter: the CTCLabelConverter of the alphabet; texts: B strings; lengths: frames per line (default T).
    Frame t covers image columns [f t, f t + f) with f = px_per_frame, or image_width // T (the model maps a line of
    width W to W // 4 tokens).  Returns per line a list of (char, x0, x1, logprob): x0 inclusive, x1 exclusive, logprob
    the sum of the character's frame log-probs.  A character outside the converter's alphabet raises ValueError;
    a line whose text cannot fit its frames raises HtrvtError."""
    if logits.dim() != 3:
        raise ValueError("logits must be [B, T, C], got shape %s" % (tuple(logits.shape),))
    B, T, _ = logits.shape
    if len(texts) != B:
        raise ValueError("%d texts for %d lines" % (len(texts), B))
    if px_per_frame is None:
        if image_width is None:
            raise ValueError("align_text needs image_width (the line image width the logits come from) or px_per_frame")
        px_per_frame = image_width // T
    ids, lens = [], []
    for text in texts:
        unknown = sorted(set(ch for ch in text if ch not in converter.dict))
        if unknown:
            raise ValueError("characters not in the converter's alphabet: %s" % ", ".join(repr(c) for c in unknown))
        ids.extend(converter.dict[ch] for ch in text)
        lens.append(len(text))
    x = logits if logits.dtype == torch.float32 else logits.float()
    if x.stride(-1) != 1:
        x = x.contiguous()
    r = ops.ctc_align(x, torch.tensor(ids, dtype=torch.int32), torch.tensor(lens, dtype=torch.int32), lengths,
                      layout="btc", is_logprob=False)
    status = r.status.cpu()
    if bool((status != 0).any()):
        raise HtrvtError("align_text: the texts of lines %s cannot be aligned to their frames (too long, status %s)"
                         % (_lines(status != 0), status[status != 0].tolist()))
    spans = r.spans.cpu().tolist()
    scores = r.token_scores.cpu().tolist()
    out = []
    for b, text in enumerate(texts):
        out.append([(ch, px_per_frame * spans[b][k][0], px_per_frame * spans[b][k][1], scores[b][k])
                    for k, ch in enumerate(text)])
    return out
