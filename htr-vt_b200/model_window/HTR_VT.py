"""`HTR_VT.create_model(nb_cls, img_size)` of the windowed variant with the reference's module surface
(model_window/model/HTR_VT.py:233-350): no absolute position embedding, a learned relative-position bias table in
every attention (`blocks.i.attn.relative_position_bias_table` [2P-1, H] + the int64 buffer
`relative_position_index` [P, P]), 16-token windowed attention in blocks 0 (shift 0) and 1 (shift 8), global
attention in the rest, no LayerNorm on the logits, and train-mode Dropout(0.1) / attention-Dropout(0.05) /
DropPath(linspace(0, 0.1, depth)).  Same state_dict keys, shapes and order as the reference (tests/golden/win_*.npz).

As in model.HTR_VT the nn.Modules are parameter containers; the arithmetic runs in the sm_100a kernels
(csrc/attention2.cu for the attention).  `set_precision("fp32")` selects the eval-mode fp32-parity forward here as
for model_v1 (csrc/exact.cu, htrvt_attention2_f32 for the attention): use it where an evaluation - greedy decode or the
LM-rescored beam - must return what the reference returns on the same weights.  Train-mode randomness: the reference draws its masks from the device
generator, so only the distribution can match - here every mask is a counter-based hash of a seed drawn per
forward from torch's CPU generator (reproducible under torch.manual_seed), regenerated in the backward.
"""
from functools import partial

import torch
import torch.nn as nn

from ..engine import Engine
from ..model.HTR_VT import MaskedAutoencoderViT as _BaseViT
from ..model.HTR_VT import _Block, _Stem  # noqa: F401


def stem_out_hw(h, w):
    """Spatial size after the truncated ResNet-18 stem (model_window/model/resnet18.py): six stride-2 steps along
    H (conv1, maxpool, layer1-3, final maxpool), two along W (layer2, layer3)."""
    for _ in range(6):
        h = (h - 1) // 2 + 1
    for _ in range(2):
        w = (w - 1) // 2 + 1
    return h, w


class _RelAttn(nn.Module):
    """Parameter container of model_window Attention (:11-31): parameter/buffer registration order matters for
    the state_dict order (own parameter, own buffer, then the child Linears)."""

    def __init__(self, dim, num_patches, num_heads):
        super().__init__()
        self.num_patches = num_patches
        self.qkv = nn.Linear(dim, 3 * dim, bias=True)
        self.proj = nn.Linear(dim, dim)
        self.relative_position_bias_table = nn.Parameter(torch.zeros(2 * num_patches - 1, num_heads))
        coords = torch.arange(num_patches)
        self.register_buffer("relative_position_index", coords[None, :] - coords[:, None] + num_patches - 1)


class _WinBlock(nn.Module):
    def __init__(self, dim, num_patches, num_heads, mlp_ratio, norm_layer):
        super().__init__()
        from ..model.HTR_VT import _Mlp
        self.norm1 = norm_layer(dim, elementwise_affine=True)
        self.attn = _RelAttn(dim, num_patches, num_heads)
        self.norm2 = norm_layer(dim, elementwise_affine=True)
        self.mlp = _Mlp(dim, int(dim * mlp_ratio))


class MaskedAutoencoderViT(_BaseViT):
    """Windowed HTR-VT encoder; constructor mirrors model_window/model/HTR_VT.py:237-246."""

    def __init__(self, nb_cls=80, img_size=[512, 32], patch_size=[8, 32], embed_dim=1024, depth=24, num_heads=16,
                 mlp_ratio=4., norm_layer=nn.LayerNorm):
        nn.Module.__init__(self)
        self.patch_embed = _Stem(embed_dim)
        self.grid_size = [img_size[0] // patch_size[0], img_size[1] // patch_size[1]]
        self.embed_dim = embed_dim
        # the reference sizes the bias table with a dummy stem pass on zeros(1, 1, img_size[1], img_size[0]) (:256-260)
        fh, fw = stem_out_hw(int(img_size[1]), int(img_size[0]))
        self.num_patches = int(fh * fw)
        self.num_heads = num_heads
        self.mask_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.drop, self.attn_drop = 0.1, 0.05
        self.drop_path = torch.linspace(0, 0.1, steps=depth).tolist()
        self.blocks = nn.ModuleList([_WinBlock(embed_dim, self.num_patches, num_heads, mlp_ratio, norm_layer)
                                     for _ in range(depth)])
        self.norm = norm_layer(embed_dim, elementwise_affine=True)
        self.head = nn.Linear(embed_dim, nb_cls)
        windows = [((16, 0) if i == 0 else ((16, 8) if i == 1 else (0, 0))) for i in range(depth)]
        eps = getattr(self.norm, "eps", 1e-6)
        self.engine = Engine(embed_dim, depth, num_heads, nb_cls, ln_eps=eps, variant="window", windows=windows)
        self.grad_sync = None
        self.dp_rank = 0
        nn.init.normal_(self.mask_token, std=.02)
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight)
                if m.bias is not None:
                    nn.init.zeros_(m.bias)

    def set_stochastic(self, drop=0.1, attn_drop=0.05, drop_path_rate=0.1):
        """Override the train-mode regularisation rates (0 everywhere makes train mode deterministic).  drop and
        attn_drop lie in [0, 1); drop_path_rate, the last block's DropPath rate, in [0, 1] (1 drops that block's
        branches for every sample)."""
        drop, attn_drop, drop_path_rate = float(drop), float(attn_drop), float(drop_path_rate)
        for name, v in (("drop", drop), ("attn_drop", attn_drop)):
            if not 0.0 <= v < 1.0:                  # (also refuses NaN)
                raise ValueError("%s must lie in [0, 1), got %r" % (name, v))
        if not 0.0 <= drop_path_rate <= 1.0:
            raise ValueError("drop_path_rate must lie in [0, 1], got %r" % drop_path_rate)
        self.drop, self.attn_drop = drop, attn_drop
        self.drop_path = torch.linspace(0, drop_path_rate, steps=len(self.blocks)).tolist()
        return self

    def _train_rng(self, batch, device):
        if self.drop <= 0 and self.attn_drop <= 0 and max(self.drop_path) <= 0:
            return None
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        gen = None
        if self.dp_rank:                            # data parallel: every rank its own dropout / DropPath stream
            seed = (seed + 0x9E3779B97F4A7C15 * self.dp_rank) % (2 ** 62)
            gen = torch.Generator().manual_seed(seed)
        dps = []
        for rate in self.drop_path:                 # timm DropPath: per-sample Bernoulli(keep) / keep
            if rate <= 0:
                dps.append((None, None))
                continue
            keep = 1.0 - rate
            pair = []
            for _ in range(2):
                kept = (torch.rand(batch, generator=gen) < keep).float()
                if keep > 0:                        # keep = 0 drops every sample: zeros, no 0 / 0 (as timm)
                    kept = kept / keep
                pair.append(kept.to(device, non_blocking=True))
            dps.append(tuple(pair))
        return {"seed": seed, "drop": self.drop, "attn_drop": self.attn_drop, "drop_path": dps}

    def forward(self, x, mask_ratio=0.0, max_span_length=1, use_masking=False, widths=None):
        T = x.shape[-1] // 4
        if T > self.num_patches:                    # model_window/model/HTR_VT.py:35-38
            raise ValueError("Sequence length N=%d exceeds configured num_patches=%d for relative bias."
                             % (T, self.num_patches))
        return super().forward(x, mask_ratio, max_span_length, use_masking, widths)


def create_model(nb_cls, img_size, **kwargs):
    """Reference factory (model_window/model/HTR_VT.py:340-350)."""
    return MaskedAutoencoderViT(nb_cls, img_size=img_size, patch_size=(4, 64), embed_dim=768, depth=4, num_heads=6,
                                mlp_ratio=4, norm_layer=partial(nn.LayerNorm, eps=1e-6), **kwargs)
