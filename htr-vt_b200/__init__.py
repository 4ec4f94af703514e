"""htr-vt_b200: B200-native (sm_100a) implementation of the HTR-VT hot path.

Line-image ViT encoder (conv stem -> LayerNorm / MHSA / GELU-MLP blocks with span masking) ->
CTC loss forward-backward -> greedy CTC decode, behind the reference's own Python surface:
  model.HTR_VT.create_model(nb_cls, img_size)      (reference model_v1/model/HTR_VT.py:244)
  CTCLoss(reduction='none', zero_infinity=True)    (reference model_v1/train.py:95)
  CTCLabelConverter(character).encode / .decode    (reference model_v1/utils/utils.py:55-86)
All device work is hand-written CUDA in csrc/ behind the C ABI declared in include/htrvt.h.
The directory name contains a hyphen; import it as `import htrvt_b200` (alias package at the repo
root) or with importlib.import_module("htr-vt_b200").
"""
from . import _lib  # noqa: F401
from .ctc import CTCLoss, ctc_loss_from_logits, greedy_decode  # noqa: F401
from .converter import CTCLabelConverter  # noqa: F401
from .metrics import ErrorRateMeter, cer_from_ids, edit_distances, format_string_for_wer  # noqa: F401
from .beam import (beam_search_with_lm_batch, ctc_lexicon_decode, ctc_lm_decode, kbest_candidates,  # noqa: F401
                   simple_ctc_beam_search_with_lm)
from .lexicon import Lexicon  # noqa: F401
from .lm import CharNGramLM  # noqa: F401
from .wordlm import WordNGramLM  # noqa: F401
from .prefetch import HostPrefetcher, RunningLoss  # noqa: F401
from .augment import SameTrCollate, augment_lines, draw_collate_params  # noqa: F401
from .align import align_text, ctc_align, forced_align  # noqa: F401

__all__ = ["CTCLoss", "ctc_loss_from_logits", "greedy_decode", "CTCLabelConverter", "ErrorRateMeter", "cer_from_ids",
           "edit_distances", "format_string_for_wer", "simple_ctc_beam_search_with_lm", "beam_search_with_lm_batch",
           "kbest_candidates", "ctc_lm_decode", "CharNGramLM", "ctc_lexicon_decode", "Lexicon", "WordNGramLM",
           "HostPrefetcher", "RunningLoss", "SameTrCollate",
           "augment_lines", "draw_collate_params", "ctc_align", "forced_align", "align_text"]
