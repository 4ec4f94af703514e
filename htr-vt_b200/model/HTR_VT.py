"""`HTR_VT.create_model(nb_cls, img_size)` with the reference's module surface
(model_v1/model/HTR_VT.py:139-254): same constructor arguments, same
`forward(x, mask_ratio=0.0, max_span_length=1, use_masking=False) -> [B, T, nb_cls]`, same
state_dict keys / shapes (SURVEY.md 8b), gradients delivered into ordinary nn.Parameter.grad.

The nn.Modules below are PARAMETER CONTAINERS only (they give the state_dict its reference names and
default initialisers); all arithmetic runs in the hand-written sm_100a kernels through engine.Engine.
There is no CPU path: calling forward on CPU tensors raises.
"""
import math
from functools import partial

import numpy as np
import torch
import torch.nn as nn

from .. import ops
from ..ddp import GradAllReduce, segment_bounds
from ..engine import Engine


def _sincos_table(embed_dim, grid_size):
    """Fixed 2-D sin/cos code over the token axis: first half of the channels encodes n % grid_w, second
    half n // grid_w, each as [sin | cos] of pos * 10000^(-k/(D/4)) (model_v1/model/HTR_VT.py:86-131)."""
    gh, gw = int(grid_size[0]), int(grid_size[1])
    n = np.arange(gh * gw)
    quarter = embed_dim // 4
    omega = 1.0 / 10000 ** (np.arange(quarter, dtype=np.float64) / quarter)
    parts = []
    for pos in ((n % gw).astype(np.float32), (n // gw).astype(np.float32)):
        ang = pos[:, None].astype(np.float64) * omega[None, :]
        parts += [np.sin(ang), np.cos(ang)]
    return torch.from_numpy(np.concatenate(parts, axis=1)).float().unsqueeze(0)


class _Residual(nn.Module):
    """Parameter container for one residual unit of the stem (names: conv1/bn1/conv2/bn2/downsample)."""

    def __init__(self, cin, cout, stride):
        super().__init__()
        self.conv1 = nn.Conv2d(cin, cout, 3, stride, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(cout, eps=1e-5)
        self.conv2 = nn.Conv2d(cout, cout, 3, 1, 1, bias=False)
        self.bn2 = nn.BatchNorm2d(cout, eps=1e-5)
        self.downsample = None
        if stride != 1 or cin != cout:
            self.downsample = nn.Sequential(nn.Conv2d(cin, cout, 1, stride, bias=False), nn.BatchNorm2d(cout, eps=1e-5))


class _Stem(nn.Module):
    """Parameter container for the truncated ResNet-18 stem (model_v1/model/resnet18.py:42-71)."""

    def __init__(self, nb_feat):
        super().__init__()
        c1, c2, c3 = nb_feat // 4, nb_feat // 2, nb_feat
        self.conv1 = nn.Conv2d(1, c1, 3, (2, 1), 1, bias=False)
        self.bn1 = nn.BatchNorm2d(c1, eps=1e-5)
        self.layer1 = nn.Sequential(_Residual(c1, c1, (2, 1)), _Residual(c1, c1, 1))
        self.layer2 = nn.Sequential(_Residual(c1, c2, 2), _Residual(c2, c2, 1))
        self.layer3 = nn.Sequential(_Residual(c2, c3, 2), _Residual(c3, c3, 1))


class _Attn(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.qkv = nn.Linear(dim, 3 * dim, bias=True)
        self.proj = nn.Linear(dim, dim)


class _Mlp(nn.Module):
    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.fc2 = nn.Linear(hidden, dim)


class _Block(nn.Module):
    def __init__(self, dim, mlp_ratio, norm_layer):
        super().__init__()
        self.norm1 = norm_layer(dim, elementwise_affine=True)
        self.attn = _Attn(dim)
        self.norm2 = norm_layer(dim, elementwise_affine=True)
        self.mlp = _Mlp(dim, int(dim * mlp_ratio))


class _EncoderFn(torch.autograd.Function):
    """Whole-encoder autograd node: forward/backward are Engine kernel schedules."""

    @staticmethod
    def forward(ctx, module, image, mask, names, save, widths, *params):
        sd = module._tensor_table()
        rng = module._train_rng(image.shape[0], image.device) if module.training else None
        logits, ectx = module.engine.forward(sd, image, mask, module.training, save, rng, widths)
        ctx.module, ctx.ectx, ctx.names, ctx.sd = module, ectx, names, sd
        ctx.shapes = [(p.shape, p.requires_grad) for p in params]
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        if ctx.ectx is None:
            raise RuntimeError("backward through a forward that did not record activations")
        module = ctx.module
        numels = [int(torch.Size(shape).numel()) for shape, _ in ctx.shapes]
        offs, split = segment_bounds(ctx.names, numels)
        flat = torch.zeros(offs[-1], dtype=torch.float32, device=dlogits.device)
        grads = {n: flat[offs[i]:offs[i] + numels[i]].view(shape)
                 for i, (n, (shape, _)) in enumerate(zip(ctx.names, ctx.shapes))}
        sync = module.grad_sync

        done = []                                        # [lo, hi) ranges of the stem segment already handed to NCCL

        def on_stage(stage):
            if sync is None:
                return
            if stage == "transformer":
                sync.reduce_async(flat[split:])          # overlaps the stem backward
            elif stage.startswith("stem:"):              # a finished stem layer: overlaps the rest of the stem backward
                pre = "patch_embed.%s." % stage[5:]
                idx = [i for i, n in enumerate(ctx.names) if n.startswith(pre)]
                if idx and offs[idx[-1] + 1] <= split:
                    sync.reduce_async(flat[offs[idx[0]]:offs[idx[-1] + 1]])
                    done.append((offs[idx[0]], offs[idx[-1] + 1]))

        module.engine.backward(ctx.sd, ctx.ectx, dlogits, grads, on_stage if sync is not None else None)
        if sync is not None:
            lo = 0
            for a, b in sorted(done) + [(split, split)]:  # what is left of the stem segment
                if a > lo:
                    sync.reduce_async(flat[lo:a])
                lo = max(lo, b)
            sync.finish()
        ctx.ectx = None
        out = tuple(grads[n] if req else None for n, (_, req) in zip(ctx.names, ctx.shapes))
        return (None, None, None, None, None, None) + out


class MaskedAutoencoderViT(nn.Module):
    """HTR-VT encoder.  Constructor mirrors the reference (model_v1/model/HTR_VT.py:143-151)."""

    def __init__(self, nb_cls=80, img_size=[512, 32], patch_size=[8, 32], embed_dim=1024, depth=24, num_heads=16,
                 mlp_ratio=4., norm_layer=nn.LayerNorm):
        super().__init__()
        self.patch_embed = _Stem(embed_dim)
        self.grid_size = [img_size[0] // patch_size[0], img_size[1] // patch_size[1]]
        self.embed_dim = embed_dim
        self.num_patches = self.grid_size[0] * self.grid_size[1]
        self.num_heads = num_heads
        self.mask_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, self.num_patches, embed_dim), requires_grad=False)
        self.blocks = nn.ModuleList([_Block(embed_dim, mlp_ratio, norm_layer) for _ in range(depth)])
        self.norm = norm_layer(embed_dim, elementwise_affine=True)
        self.head = nn.Linear(embed_dim, nb_cls)
        eps = getattr(self.norm, "eps", 1e-6)
        self.engine = Engine(embed_dim, depth, num_heads, nb_cls, ln_eps=eps, variant="v1")
        self.grad_sync = None           # set by enable_data_parallel(): NCCL all-reduce inside backward
        self.dp_rank = 0
        self._init_parameters()

    def _init_parameters(self):
        self.pos_embed.data.copy_(_sincos_table(self.embed_dim, self.grid_size))
        nn.init.normal_(self.mask_token, std=.02)
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight)
                if m.bias is not None:
                    nn.init.zeros_(m.bias)

    # -- plumbing -------------------------------------------------------------------------------
    def _train_rng(self, batch, device):
        """Stochastic-regularisation state of one train-mode forward (None: model_v1 has no dropout / DropPath)."""
        return None

    def _slots(self):
        """(full name, owning module, key, is_parameter) of every parameter and buffer, in named_parameters() /
        named_buffers() order.  The module tree is fixed after construction, so the walk is done once; the tensors are
        looked up in their owners' dicts every forward (`.to()` / `load_state_dict(assign=True)` may replace them)."""
        slots = self.__dict__.get("_slot_cache")
        if slots is None:
            slots = []
            for prefix, mod in self.named_modules():
                for key in mod._parameters:
                    if mod._parameters[key] is not None:
                        slots.append((prefix + "." + key if prefix else key, mod, key, True))
            for prefix, mod in self.named_modules():
                for key in mod._buffers:
                    if mod._buffers[key] is not None:
                        slots.append((prefix + "." + key if prefix else key, mod, key, False))
            self.__dict__["_slot_cache"] = slots
        return slots

    def _tensor_table(self):
        return {name: (mod._parameters[key] if is_p else mod._buffers[key]) for name, mod, key, is_p in self._slots()}

    def set_precision(self, precision):
        """"bf16" (default): 16-bit tensor-core operands, fp32 accumulation - the product path.  "fp32": eval-mode
        parity forward (fp32 tensors, split-bf16 contractions): logits within 1e-4 of the fp32 reference and greedy
        decode strings identical to it (north_star); forward only, under model.eval() + torch.no_grad().  Both
        variants: model_v1 and the windowed model (model_window), whose fp32 attention keeps its relative-position
        bias, shifted 16-token windows and padded lines."""
        if precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        self.engine.precision = precision
        return self

    def enable_data_parallel(self, group=None, broadcast=True):
        """Average gradients over the ranks of `group` inside backward (batch sharding, one process per GPU).
        Like torch DDP, every parameter and buffer is first broadcast from rank 0, so replicas start identical even
        when the ranks were seeded differently (e.g. for augmentation).  Randomness under DP: the span mask comes from
        torch's CPU generator exactly as in the reference (ranks with the same seed draw the same mask, differently
        seeded ranks different ones - both are faithful, the reference draws a fresh mask per forward);
        the window variant's dropout / DropPath streams are offset by the rank so that no two ranks share a mask."""
        import torch.distributed as dist
        from ..ddp import broadcast_tensors
        self.grad_sync = GradAllReduce(group)
        self.dp_rank = dist.get_rank(group) if (dist.is_available() and dist.is_initialized()) else 0
        if broadcast:
            broadcast_tensors(list(self._tensor_table().values()), group, src=0)
            ops.weights_changed()
        return self

    def __deepcopy__(self, memo):           # EMA deep-copies the model (utils.py:130): keep comm objects shared
        import copy
        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k == "_slot_cache":
                continue                    # holds references to THIS tree's modules
            new.__dict__[k] = v if k == "grad_sync" else copy.deepcopy(v, memo)
        return new

    @staticmethod
    def span_mask(L, mask_ratio, max_span_length):
        """Same draws, in the same order, from the CPU default generator as the reference's
        generate_span_mask (model_v1/model/HTR_VT.py:202-210): int(L*ratio)//span spans, one mask per batch."""
        mask = torch.ones(L)
        for _ in range(int(L * mask_ratio) // max_span_length):
            idx = int(torch.randint(L - max_span_length, (1,)))
            mask[idx:idx + max_span_length] = 0
        return mask

    def forward(self, x, mask_ratio=0.0, max_span_length=1, use_masking=False, widths=None):
        """Reference signature (model_v1/model/HTR_VT.py:222).  x: fp32 [B,1,H,W] in [0,1] as the reference's loader
        produces it - or the SAME images still as uint8 (value = round(255 x), padding 255): one kernel then does
        /255, pad-to-W with 1.0 for columns >= widths[b] (optional) and the input LayerNorm (SURVEY.md 8f row 2)."""
        if not x.is_cuda:
            raise ops.HtrvtError("htr-vt_b200 MaskedAutoencoderViT.forward needs CUDA tensors (no CPU fallback)")
        if x.shape[-1] % 4:
            raise ValueError("line image width must be a multiple of 4 (the stem halves the width twice; got %d)"
                             % x.shape[-1])
        mask = None
        if use_masking:
            L = x.shape[-1] // 4                 # tokens = stem output columns (exact: the width is a multiple of 4)
            mask = self.span_mask(L, mask_ratio, max_span_length).to(x.device, non_blocking=True)
        names, params = zip(*[(name, mod._parameters[key]) for name, mod, key, is_p in self._slots() if is_p])
        save = torch.is_grad_enabled() and any(p.requires_grad for p in params)
        return _EncoderFn.apply(self, x, mask, names, save, widths, *params)


def create_model(nb_cls, img_size, **kwargs):
    """Reference factory (model_v1/model/HTR_VT.py:244-254): fixed architecture hyper-parameters."""
    return MaskedAutoencoderViT(nb_cls, img_size=img_size, patch_size=(4, 64), embed_dim=768, depth=4, num_heads=6,
                                mlp_ratio=4, norm_layer=partial(nn.LayerNorm, eps=1e-6), **kwargs)
