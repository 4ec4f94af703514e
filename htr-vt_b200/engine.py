"""Forward / backward schedule of the HTR-VT encoder on the sm_100a kernels.

One explicit kernel sequence (no autograd graph inside): forward() records the activations the
backward needs in a context, backward() walks the layers in reverse and writes fp32 gradients for
every trainable parameter.  Data layout in HBM:
  * stem activations   NHWC bf16 (channels innermost => the implicit-GEMM A operand is a TMA box);
  * token stream       fp32 [B*T, D] residual, bf16 copies only as GEMM operands;
  * weights            fp32 masters in the nn.Parameters (reference layouts: OIHW, [out,in]);
                       bf16 operand copies ([Cout, taps, Cin] / [out, in]) are re-packed every forward,
                       because SAM perturbs the masters in place twice per iteration (SURVEY.md 9.19).
Reference semantics: model_v1/model/HTR_VT.py:222-241 and model_v1/model/resnet18.py:73-84.
"""
import os

import torch

from . import ops

STEM_LAYERS = (("layer1", (2, 1)), ("layer2", (2, 2)), ("layer3", (2, 2)))
# BatchNorm-backward reduction in the epilogue of the GEMM that produces the gradient (HTRVT_FUSE_BN_BWD=0: two-pass route)
FUSE_BN_BWD = os.environ.get("HTRVT_FUSE_BN_BWD", "1") != "0"
# Weight-gradient GEMMs on a second stream (HTRVT_WGRAD_STREAM=0: everything on the caller's stream).  They depend only on
# a layer's dY and its saved input, nothing in the backward reads them before the gradients are handed over, so they fill
# the SMs the input-gradient chain leaves idle: kernel tails, grids smaller than the machine, and the HBM-bound
# BatchNorm / LayerNorm passes whose CTAs fit beside a resident GEMM CTA.
WGRAD_STREAM = os.environ.get("HTRVT_WGRAD_STREAM", "1") != "0"


class _SideStream(object):
    """Runs independent launches of the backward on a per-device second stream.  Every submission waits for what the
    caller's stream has enqueued so far (its inputs were produced there); `join()` makes the caller's stream wait for
    the side work and only then drops the references that kept the inputs' memory from being reused."""
    _streams = {}

    def __init__(self, device, enabled):
        self.on = bool(enabled) and device.type == "cuda"
        self.keep = []
        self.pending = False
        if self.on:
            key = device.index if device.index is not None else torch.cuda.current_device()
            st = _SideStream._streams.get(key)
            if st is None:
                st = _SideStream._streams[key] = (torch.cuda.Stream(device=device), torch.cuda.Event())
            self.side, self.ev = st
            self.main = torch.cuda.current_stream(device)

    def run(self, fn, *args):
        if not self.on:
            return fn(*args)
        self.ev.record(self.main)
        self.side.wait_event(self.ev)
        self.keep.append(args)
        self.pending = True
        with torch.cuda.stream(self.side):
            return fn(*args)

    def join(self):
        if self.on and self.pending:
            self.main.wait_stream(self.side)
            self.pending = False
        self.keep = []


class _Ctx(object):
    pass


def _bn_args(sd, prefix):
    return (sd[prefix + ".weight"], sd[prefix + ".bias"], sd[prefix + ".running_mean"], sd[prefix + ".running_var"],
            sd[prefix + ".num_batches_tracked"])


class Engine(object):
    """Stateless w.r.t. parameters: every call receives the module's current tensors by name."""

    def __init__(self, embed_dim, depth, num_heads, nb_cls, ln_eps=1e-6, variant="v1", windows=None):
        self.D, self.depth, self.H, self.C = embed_dim, depth, num_heads, nb_cls
        self.hd = embed_dim // num_heads
        self.ln_eps = ln_eps
        self.variant = variant
        # window variant: (window_size, shift) per block (model_window/model/HTR_VT.py:274-275)
        self.windows = list(windows) if windows is not None else [(0, 0)] * depth
        # "bf16": 16-bit tensor-core operands (the product path); "fp32": the fp32-parity eval forward (split-bf16
        # operands, fp32 everywhere else - csrc/exact.cu), logits within 1e-4 of the fp32 reference
        self.precision = "bf16"
        if self.hd != 128:
            raise ops.HtrvtError("attention kernel is specialised for head_dim 128 (got %d)" % self.hd)
        if embed_dim % 256 or nb_cls < 2:
            raise ops.HtrvtError("embed_dim must be a multiple of 256")

    # ------------------------------------------------------------------------------------------
    def _bn(self, sd, prefix, partial, count, training):
        g, b, rm, rv, nbt = _bn_args(sd, prefix)
        return ops.bn_finalize(partial if training else None, count, g, b, rm, rv, nbt, training)

    def _conv(self, x, wp, ks, stride, training, pool=None):
        N, H, W, _ = x.shape
        stats = None
        if training:
            rows = ops.conv_stats_rows(N, H, W, ks, stride[0], stride[1])
            n = rows * 2 * wp.shape[0]                                         # one [2, Cout] row per CTA quadrant
            if pool is not None and pool[1] + n <= pool[0].numel():
                stats = pool[0][pool[1]:pool[1] + n].view(rows, 2, wp.shape[0])
                pool[1] += n
            else:
                stats = torch.zeros((rows, 2, wp.shape[0]), dtype=torch.float32, device=x.device)
        y = ops.conv_fwd(x, wp, ks, stride[0], stride[1], stats=stats)
        return y, stats

    def forward(self, sd, image, mask, training, save, rng=None, widths=None):
        """sd: name -> tensor (parameters + BN buffers); image fp32 [B,1,H,W] in [0,1], or the loader's uint8 line
        images [B,1,H,W] (value / 255, columns >= widths[b] read as padding 1.0: dataset.py:13-45,129-130) which one
        kernel converts, pads and normalises; mask fp32 [T] or None.
        rng (window variant, train mode): dict(seed, drop, attn_drop, drop_path=[(dp1, dp2) per block]) or None.
        Returns (logits fp32 [B,T,C], ctx | None)."""
        if image.dim() != 4 or image.shape[1] != 1:
            raise ValueError("expected image [B, 1, H, W]")
        if not image.is_cuda:
            raise ops.HtrvtError("htr-vt_b200 runs on CUDA only (no CPU fallback)")
        if self.precision == "fp32":
            if training or save:
                raise ops.HtrvtError("precision='fp32' is the eval-mode parity forward: call model.eval() and run under "
                                     "torch.no_grad() (training runs with 16-bit tensor-core operands)")
            return self.forward_fp32(sd, image, mask, widths), None
        B, _, Hi, Wi = image.shape
        D, C = self.D, self.C
        ctx = _Ctx() if save else None
        u8 = image.dtype == torch.uint8
        if not u8:
            image = image.contiguous().float()

        # ---- weights: bf16 operand copies -----------------------------------------------------
        names, items = [], []
        for k, v in sd.items():
            if k.startswith("patch_embed.") and k.endswith("weight") and v.dim() == 4 and v.shape[1] > 1:
                names.append(k)
                items.append((v, "conv"))
                if save:                          # [Cin, taps, Cout] copy: K-major B operand of the input-gradient GEMM
                    names.append("T:" + k)
                    items.append((v, "convT"))
            elif v.dim() == 2 and k.endswith(".weight"):
                names.append(k)
                items.append((v, "cast"))
        C8 = (C + 7) // 8 * 8            # the head GEMM runs on a class axis padded to a multiple of 8 (zero rows)
        # eval mode: the packed copies are reused while no parameter changed (autograd version counters + the epoch
        # our own raw-pointer optimizer kernels bump); train mode repacks every forward (SAM rewrites the weights)
        # Eval mode also FOLDS each block's bn1 into conv1 (running statistics: w' = w * scale[co] in the repack, shift + ReLU
        # in the conv epilogue), so that BatchNorm pass disappears, and keeps every BN's affine coefficients in the cache.
        fold = not training and not save
        key = bnst = None
        if fold:
            stem = [v for k, v in sd.items() if k.startswith("patch_embed.")]
            key = (ops.WEIGHT_EPOCH, tuple((v.data_ptr(), v._version) for v, _ in items),
                   tuple((v.data_ptr(), v._version) for v in stem))
        pack_side = None
        cached = getattr(self, "_wp_cache", None)
        if key is not None and cached is not None and cached[0] == key:
            wp, bnst = cached[1], cached[2]
        else:
            if fold:
                bnst = {k[:-len(".running_mean")]: self._bn(sd, k[:-len(".running_mean")], None, 1, False)
                        for k in sd if k.startswith("patch_embed.") and k.endswith(".running_mean")}
                def bn_of(n):                     # conv parameter name -> the BatchNorm that follows it
                    if n.endswith(".downsample.0.weight"):
                        return n[:-len("0.weight")] + "1"
                    return n[:-len(".convX.weight")] + ".bn" + n[-len("X.weight")]
                items = [(v, kind, bnst[bn_of(n)][2]) if kind == "conv" else (v, kind)
                         for n, (v, kind) in zip(names, items)]
            # train mode: the ~50 packed tensors of the previous step are overwritten in place when no recorded forward
            # still waits for its backward (stream order protects the kernels already enqueued); a second forward before
            # the first one's backward (gradient accumulation over graphs) gets fresh tensors
            sig = (tuple(names), tuple(v.data_ptr() for v, *_ in items), str(image.device))
            pool = getattr(self, "_wp_pool", None)
            reuse = None
            if not fold and pool is not None and pool[0] == sig and getattr(self, "_wp_busy", 0) == 0:
                reuse = pool[1]
            # steady-state train steps (in-place re-pack, no allocation): the pack runs on the side stream under the
            # stem head, which reads conv1's fp32 weights only; joined in front of the first stem block
            pack_side = _SideStream(image.device, WGRAD_STREAM and reuse is not None)
            packed = pack_side.run(lambda: ops.pack_weights(
                items, pad_rows={"head.weight": C8} if C8 != C else None, names=names,
                reuse=reuse))                                       # one launch for all 36 weight tensors
            wp = dict(zip(names, packed))
            if not fold:
                self._wp_pool = (sig, packed)
            self._wp_cache = (key, wp, bnst) if key is not None else None
        if save:
            self._wp_busy = getattr(self, "_wp_busy", 0) + 1          # released by backward()

        # ---- stem -----------------------------------------------------------------------------
        if u8:
            x0, _, _ = ops.line_prep_u8(image[:, 0], widths, 1e-5)
        else:
            x0, _, _ = ops.sample_ln_fwd(image.view(B, Hi, Wi), torch.float32, 1e-5)
        # stem head (conv1 -> bn1 -> relu -> maxpool) fused: the K = 9 conv output is never materialised
        w1 = sd["patch_embed.conv1.weight"]
        moments = part = None
        if training:
            moments, part = ops.stem_head_moments(x0, w1)
        st1 = bnst["patch_embed.bn1"] if fold else self._bn(sd, "patch_embed.bn1", part, B * (Hi // 2) * Wi, training)
        # forward stem tensors are fp16 (ops.STEM_DTYPE); with `save` every activation that feeds a convolution also
        # gets a bf16 copy (x_bf / a1_bf) from the kernel that writes it: the weight-gradient GEMMs need the format of dY
        x_bf = None
        if save:
            x, code1, x_bf = ops.stem_head_fwd(x0, w1, st1, True, want_bf16=True)
        else:
            x, code1 = ops.stem_head_fwd(x0, w1, st1, False)
        if pack_side is not None:
            pack_side.join()
        blocks = []
        last_block = "patch_embed.%s.1" % STEM_LAYERS[-1][0]
        zpool = None
        if training:            # one memset for the statistics partials of all 15 stem convolutions
            rows = ops.conv_stats_rows(B, Hi, Wi, 3, 1, 1)
            total = sum(rows * 2 * v.shape[0] for k, v in wp.items() if k.startswith("patch_embed."))
            zpool = [torch.zeros(total, dtype=torch.float32, device=image.device), 0]
        for lname, stride in STEM_LAYERS:
            for bi in range(2):
                p = "patch_embed.%s.%d" % (lname, bi)
                s = stride if bi == 0 else (1, 1)
                if fold:
                    # every BatchNorm of the block is folded (scale in the weights, shift as an epilogue bias): conv1
                    # writes relu(bn1(conv1 x)), the 1x1 downsample writes bn_d(ds x), conv2's epilogue adds the skip
                    # connection and applies the ReLU - three kernels per block, no BatchNorm pass
                    a1 = ops.conv_fwd(x, wp[p + ".conv1.weight"], 3, s[0], s[1], relu=True, bias=bnst[p + ".bn1"][3])
                    skip = x
                    if (p + ".downsample.0.weight") in sd:
                        skip = ops.conv_fwd(x, wp[p + ".downsample.0.weight"], 1, s[0], s[1],
                                            bias=bnst[p + ".downsample.1"][3])
                    x = ops.conv_fwd(a1, wp[p + ".conv2.weight"], 3, 1, 1, relu=True, bias=bnst[p + ".bn2"][3], res=skip)
                    continue
                else:
                    r1, pt1 = self._conv(x, wp[p + ".conv1.weight"], 3, s, training, zpool)
                    cnt = r1.numel() // r1.shape[-1]
                    sa = self._bn(sd, p + ".bn1", pt1, cnt, training)
                    a1_bf = None
                    if save:
                        a1, k1, a1_bf = ops.bn_act_fwd(r1, sa, True, want_mask=True, want_bf16=True)
                    else:
                        a1, k1 = ops.bn_act_fwd(r1, sa, True), None
                    r2, pt2 = self._conv(a1, wp[p + ".conv2.weight"], 3, (1, 1), training, zpool)
                    sb = self._bn(sd, p + ".bn2", pt2, cnt, training)
                rd = sdn = None
                if (p + ".downsample.0.weight") in sd:
                    rd, ptd = self._conv(x, wp[p + ".downsample.0.weight"], 1, s, training, zpool)
                    sdn = bnst[p + ".downsample.1"] if fold else self._bn(sd, p + ".downsample.1", ptd, cnt, training)
                    y = ops.bn_act_fwd(r2, sb, True, raw2=rd, st2=sdn, want_mask=save,
                                       want_bf16=save and p != last_block)
                else:
                    y = ops.bn_act_fwd(r2, sb, True, res=x, want_mask=save, want_bf16=save and p != last_block)
                k2 = y_bf = None
                if save:
                    if p != last_block:
                        y, k2, y_bf = y
                    else:
                        y, k2 = y
                    # the backward reads the bf16 copies (weight gradients) and the raw conv outputs / mask bits
                    # (BatchNorm backward); the fp16 activations are not kept
                    blocks.append((p, s, x_bf, r1, sa, a1_bf, k1, r2, sb, rd, sdn, k2))
                x, x_bf = y, y_bf
        Bx, Hx, Wx, Cx = x.shape
        tok, idx2 = ops.pool_fwd(x, None, save)                  # [B, Hx/2, T, D]
        if tok.shape[1] != 1 or Cx != D:
            raise ValueError("stem output height must pool to 1 (image height 64)")
        T = Wx
        M = B * T

        # ---- tokens ---------------------------------------------------------------------------
        pos = sd.get("pos_embed")
        if pos is not None and pos.shape[1] != T:
            raise ValueError("pos_embed has %d positions, sequence has %d" % (pos.shape[1], T))
        xs = ops.tokens_fwd(tok, mask, sd["mask_token"], pos, B, T, D)
        scale = self.hd ** -0.5
        tblocks = []
        pend = None                       # bf16 GEMM output still to be added to the residual stream
        drop = rng["drop"] if rng else 0.0
        attn_drop = rng["attn_drop"] if rng else 0.0
        seed = rng["seed"] if rng else 0
        for i in range(self.depth):
            p = "blocks.%d" % i
            dp1, dp2 = rng["drop_path"][i] if rng else (None, None)
            # x1 = xs + pend (previous block's fc2 output), h1 = LN1(x1): the residual add is fused into the LN
            h1, m1, r1s, x1 = ops.row_ln_fwd(xs, sd[p + ".norm1.weight"], sd[p + ".norm1.bias"], self.ln_eps, pend)
            qkv = torch.empty((M, 3 * D), dtype=torch.bfloat16, device=xs.device)
            ops.gemm_tn(h1, wp[p + ".attn.qkv.weight"], qkv, bias=sd[p + ".attn.qkv.bias"])
            o = torch.empty((M, D), dtype=torch.bfloat16, device=xs.device)
            lse = torch.empty((B, self.H, T), dtype=torch.float32, device=xs.device)
            if self.variant == "v1":
                ops.attention_fwd(qkv.view(B, T, 3, self.H, self.hd), o.view(B, T, D), lse, scale)
            else:
                tbl = sd[p + ".attn.relative_position_bias_table"]
                ws, sh = self.windows[i]
                ops.attention2_fwd(qkv.view(B, T, 3, self.H, self.hd), o.view(B, T, D), lse, scale, tbl,
                                   (tbl.shape[0] + 1) // 2, ws, sh, attn_drop, seed + 16 * i)
            y1 = torch.empty((M, D), dtype=torch.bfloat16, device=xs.device)
            ops.gemm_tn(o, wp[p + ".attn.proj.weight"], y1, bias=sd[p + ".attn.proj.bias"])
            if rng:
                ops.dropout_(y1, T * D, drop, seed, 8 * i + 1, dp1)
            h2, m2, r2s, x2 = ops.row_ln_fwd(x1, sd[p + ".norm2.weight"], sd[p + ".norm2.bias"], self.ln_eps, y1)
            hid = wp[p + ".mlp.fc1.weight"].shape[0]
            # timm Mlp: fc1 -> nn.GELU in ONE kernel (GELU in the GEMM epilogue); with `save` the epilogue also stores
            # u = gelu'(pre-activation) (a second TMA store per box): the backward multiplies by it
            a = torch.empty((M, hid), dtype=torch.bfloat16, device=xs.device)
            u = torch.empty((M, hid), dtype=torch.bfloat16, device=xs.device) if save else None
            ops.gemm_tn(h2, wp[p + ".mlp.fc1.weight"], a, bias=sd[p + ".mlp.fc1.bias"], gelu=True, pre=u)
            if rng:
                ops.dropout_(a, T * hid, drop, seed, 8 * i + 2)
            y2 = torch.empty((M, D), dtype=torch.bfloat16, device=xs.device)
            ops.gemm_tn(a, wp[p + ".mlp.fc2.weight"], y2, bias=sd[p + ".mlp.fc2.bias"])
            if rng:
                ops.dropout_(y2, T * D, drop, seed, 8 * i + 3, dp2)
            if save:
                tblocks.append((i, p, x1, h1, m1, r1s, qkv, o, lse, x2, h2, m2, r2s, a, u))
            xs, pend = x2, y2
        hf, mf, rf, xs = ops.row_ln_fwd(xs, sd["norm.weight"], sd["norm.bias"], self.ln_eps, pend)
        raw_logits = torch.empty((M, C8), dtype=torch.float32, device=xs.device)
        hb = sd["head.bias"] if C8 == C else torch.nn.functional.pad(sd["head.bias"].detach(), (0, C8 - C))
        ops.gemm_tn(hf, wp["head.weight"], raw_logits, bias=hb)
        if C8 != C:
            raw_logits = raw_logits[:, :C].contiguous()
        if self.variant == "v1":
            logits, _, rl = ops.sample_ln_fwd(raw_logits.view(B, T, C), torch.float32, 1e-5)
        else:
            logits, rl = raw_logits.view(B, T, C), None
        if save:
            ctx.B, ctx.T, ctx.Hi, ctx.Wi = B, T, Hi, Wi
            ctx.wp, ctx.x0, ctx.moments, ctx.st1, ctx.code1 = wp, x0, moments, st1, code1
            ctx.blocks, ctx.l3_shape, ctx.idx2, ctx.mask = blocks, (Bx, Hx, Wx, Cx), idx2, mask
            ctx.tblocks, ctx.x_final, ctx.hf, ctx.mf, ctx.rf = tblocks, xs, hf, mf, rf
            ctx.logits, ctx.rl, ctx.rng = logits, rl, rng
        return logits, ctx

    # ------------------------------------------------------------------------------------------
    def _planes_fp32(self, sd):
        """bf16 plane triples of every GEMM weight (conv weights as [Cout, taps, Cin]; head padded to 8 classes),
        cached while no parameter changes."""
        key = (ops.WEIGHT_EPOCH, tuple((v.data_ptr(), v._version) for v in sd.values()))
        cached = getattr(self, "_fp32_cache", None)
        if cached is not None and cached[0] == key:
            return cached[1]
        wp = {}
        C8 = (self.C + 7) // 8 * 8
        for k, v in sd.items():
            if k.startswith("patch_embed.") and k.endswith("weight") and v.dim() == 4 and v.shape[1] > 1:
                co, ci, kh, kw = v.shape
                wp[k] = ops.split3(v.detach().permute(0, 2, 3, 1).reshape(co, kh * kw, ci))
            elif v.dim() == 2 and k.endswith(".weight"):
                w = v.detach()
                if k == "head.weight" and C8 != self.C:
                    w = torch.nn.functional.pad(w, (0, 0, 0, C8 - self.C))
                wp[k] = ops.split3(w)
        bn = {k[:-len(".running_mean")]: self._bn(sd, k[:-len(".running_mean")], None, 1, False)
              for k in sd if k.startswith("patch_embed.") and k.endswith(".running_mean")}
        self._fp32_cache = (key, (wp, bn))
        return wp, bn

    def forward_fp32(self, sd, image, mask=None, widths=None, chunk=32):
        """Eval-mode forward with fp32 tensors between kernels and split-bf16 tensor-core contractions (csrc/exact.cu;
        model_v1/model/HTR_VT.py:222-241, model_window/model/HTR_VT.py:320-337, model_v1/model/resnet18.py:73-84 with
        running statistics).  -> logits fp32 [B, T, C]."""
        if image.shape[0] > chunk:                      # fp32 activations: bound the working set
            return torch.cat([self.forward_fp32(sd, image[i:i + chunk], mask,
                                                None if widths is None else widths[i:i + chunk], chunk)
                              for i in range(0, image.shape[0], chunk)])
        wp, bn = self._planes_fp32(sd)
        B, _, Hi, Wi = image.shape
        D, C = self.D, self.C
        if image.dtype == torch.uint8:
            x0, _, _ = ops.line_prep_u8(image[:, 0], widths, 1e-5)
        else:
            x0, _, _ = ops.sample_ln_fwd(image.contiguous().float().view(B, Hi, Wi), torch.float32, 1e-5)
        x, _ = ops.stem_head_fwd(x0, sd["patch_embed.conv1.weight"], bn["patch_embed.bn1"], False,
                                 out_dtype=torch.float32)
        xp = ops.split3(x)
        for lname, stride in STEM_LAYERS:
            for bi in range(2):
                p = "patch_embed.%s.%d" % (lname, bi)
                s = stride if bi == 0 else (1, 1)
                r1 = ops.conv_fwd_split(xp, wp[p + ".conv1.weight"], 3, s[0], s[1])
                _, a1p = ops.bn_act_f32(r1, bn[p + ".bn1"], True, want_y=False)
                r2 = ops.conv_fwd_split(a1p, wp[p + ".conv2.weight"], 3, 1, 1)
                if (p + ".downsample.0.weight") in sd:
                    rd = ops.conv_fwd_split(xp, wp[p + ".downsample.0.weight"], 1, s[0], s[1])
                    x, xp = ops.bn_act_f32(r2, bn[p + ".bn2"], True, raw2=rd, st2=bn[p + ".downsample.1"])
                else:
                    x, xp = ops.bn_act_f32(r2, bn[p + ".bn2"], True, res=x)
        tok = ops.maxpool_f32(x)
        if tok.shape[1] != 1 or tok.shape[3] != D:
            raise ValueError("stem output height must pool to 1 (image height 64)")
        T = tok.shape[2]
        M = B * T
        pos = sd.get("pos_embed")
        if pos is not None and pos.shape[1] != T:
            raise ValueError("pos_embed has %d positions, sequence has %d" % (pos.shape[1], T))
        xs = ops.tokens_f32(tok, mask, sd["mask_token"], pos, B, T, D)
        dev = xs.device
        pend = None
        for i in range(self.depth):
            p = "blocks.%d" % i
            h1p, x1 = ops.row_ln_f32(xs, sd[p + ".norm1.weight"], sd[p + ".norm1.bias"], self.ln_eps, pend)
            qkv = torch.empty((M, 3 * D), dtype=torch.float32, device=dev)
            ops.gemm_tn_split(h1p, wp[p + ".attn.qkv.weight"], qkv, sd[p + ".attn.qkv.bias"])
            if self.variant == "v1":
                o = ops.attention_f32(qkv, B, self.H, T, self.hd, self.hd ** -0.5)
            else:
                tbl = sd[p + ".attn.relative_position_bias_table"]
                ws, sh = self.windows[i]
                o = ops.attention2_f32(qkv, B, self.H, T, self.hd, self.hd ** -0.5, tbl, (tbl.shape[0] + 1) // 2, ws, sh)
            op = ops.split3(o)
            y1 = torch.empty((M, D), dtype=torch.float32, device=dev)
            ops.gemm_tn_split(op, wp[p + ".attn.proj.weight"], y1, sd[p + ".attn.proj.bias"])
            h2p, x2 = ops.row_ln_f32(x1, sd[p + ".norm2.weight"], sd[p + ".norm2.bias"], self.ln_eps, y1)
            u = torch.empty((M, wp[p + ".mlp.fc1.weight"].shape[1]), dtype=torch.float32, device=dev)
            ops.gemm_tn_split(h2p, wp[p + ".mlp.fc1.weight"], u, sd[p + ".mlp.fc1.bias"])
            y2 = torch.empty((M, D), dtype=torch.float32, device=dev)
            ops.gemm_tn_split(ops.gelu_split(u), wp[p + ".mlp.fc2.weight"], y2, sd[p + ".mlp.fc2.bias"])
            xs, pend = x2, y2
        hfp, _ = ops.row_ln_f32(xs, sd["norm.weight"], sd["norm.bias"], self.ln_eps, pend)
        C8 = (C + 7) // 8 * 8
        raw_logits = torch.empty((M, C8), dtype=torch.float32, device=dev)
        hb = sd["head.bias"] if C8 == C else torch.nn.functional.pad(sd["head.bias"].detach(), (0, C8 - C))
        ops.gemm_tn_split(hfp, wp["head.weight"], raw_logits, hb)
        if C8 != C:
            raw_logits = raw_logits[:, :C].contiguous()
        if self.variant != "v1":                        # the windowed variant has no LayerNorm on the logits
            return raw_logits.view(B, T, C)
        logits, _, _ = ops.sample_ln_fwd(raw_logits.view(B, T, C), torch.float32, 1e-5)
        return logits

    # ------------------------------------------------------------------------------------------
    def backward(self, sd, ctx, dlogits, grads, on_stage=None):
        """dlogits fp32 [B,T,C]; grads: name -> fp32 tensor (accumulated into, +=)."""
        if ctx.moments is None:
            # an eval-mode forward normalised with the running statistics: the BatchNorm backward kernels differentiate
            # through BATCH statistics, so refuse before any gradient is written (INTEGRATION.md, limits)
            raise ops.HtrvtError("backward needs a train-mode forward (batch statistics)")
        B, T, D, C = ctx.B, ctx.T, self.D, self.C
        M = B * T
        wp = ctx.wp
        dev = dlogits.device
        side = _SideStream(dev, WGRAD_STREAM)
        dlogits = dlogits.contiguous().float()
        ldc = (C + 7) // 8 * 8
        if self.variant == "v1":
            draw = ops.sample_ln_bwd(dlogits, ctx.logits, ctx.rl, C, ldc)          # bf16 [M, ldc], pad columns zero
        else:
            draw = torch.zeros((M, ldc), dtype=torch.bfloat16, device=dev)
            draw[:, :C] = ops.cast_bf16(dlogits.view(M, C))
        if ldc == C:
            side.run(ops.linear_wgrad, draw, ctx.hf, grads["head.weight"])
            ops.colsum_bf16(draw, grads["head.bias"])
        else:                            # class axis padded to a multiple of 8: gradients of the zero rows are dropped
            gw = torch.zeros((ldc, D), dtype=torch.float32, device=dev)
            gb = torch.zeros(ldc, dtype=torch.float32, device=dev)
            ops.linear_wgrad(draw, ctx.hf, gw)
            ops.colsum_bf16(draw, gb)
            grads["head.weight"] += gw[:C]
            grads["head.bias"] += gb[:C]
        dhf = torch.empty((M, D), dtype=torch.bfloat16, device=dev)
        ops.gemm_nn(draw, wp["head.weight"], dhf)
        gx = torch.empty((M, D), dtype=torch.float32, device=dev)
        ops.row_ln_bwd(dhf, ctx.x_final, ctx.mf, ctx.rf, sd["norm.weight"], gx, False, grads["norm.weight"],
                       grads["norm.bias"])
        scale = self.hd ** -0.5
        rng = ctx.rng
        drop = rng["drop"] if rng else 0.0
        attn_drop = rng["attn_drop"] if rng else 0.0
        seed = rng["seed"] if rng else 0
        for (i, p, x1, h1, m1, r1s, qkv, o, lse, x2, h2, m2, r2s, a, u) in reversed(ctx.tblocks):
            dp1, dp2 = rng["drop_path"][i] if rng else (None, None)
            hid = a.shape[1]
            if rng and (drop > 0.0 or dp2 is not None):   # same counter-based masks as the forward
                gy = ops.cast_bf16(gx)
                ops.dropout_(gy, T * D, drop, seed, 8 * i + 3, dp2)
                ops.colsum_bf16(gy, grads[p + ".mlp.fc2.bias"])
            else:                        # bf16 dY of fc2 and fc2's bias gradient in one pass over the residual gradient
                gy = ops.cast_colsum_bf16(gx, grads[p + ".mlp.fc2.bias"])
            side.run(ops.linear_wgrad, gy, a, grads[p + ".mlp.fc2.weight"])
            fused_bias = False
            if rng and drop > 0.0:       # dropout sits between the activation and fc2: its mask applies to da first
                da = torch.empty_like(a)
                ops.gemm_nn(gy, wp[p + ".mlp.fc2.weight"], da)
                ops.dropout_(da, T * hid, drop, seed, 8 * i + 2)
                du = ops.mul_bf16(da, u)             # u holds gelu'(pre-activation)
            else:                        # fc2's input gradient and the activation's backward in one kernel
                du = torch.empty_like(a)
                ops.gemm_nn(gy, wp[p + ".mlp.fc2.weight"], du, gelu_u=u, colsum=grads[p + ".mlp.fc1.bias"])
                fused_bias = True
            side.run(ops.linear_wgrad, du, h2, grads[p + ".mlp.fc1.weight"])
            if not fused_bias:
                ops.colsum_bf16(du, grads[p + ".mlp.fc1.bias"])
            dh2 = torch.empty((M, D), dtype=torch.bfloat16, device=dev)
            ops.gemm_nn(du, wp[p + ".mlp.fc1.weight"], dh2)
            ops.row_ln_bwd(dh2, x2, m2, r2s, sd[p + ".norm2.weight"], gx, True, grads[p + ".norm2.weight"],
                           grads[p + ".norm2.bias"])
            if rng and (drop > 0.0 or dp1 is not None):
                gy = ops.cast_bf16(gx)
                ops.dropout_(gy, T * D, drop, seed, 8 * i + 1, dp1)
                ops.colsum_bf16(gy, grads[p + ".attn.proj.bias"])
            else:
                gy = ops.cast_colsum_bf16(gx, grads[p + ".attn.proj.bias"])
            side.run(ops.linear_wgrad, gy, o, grads[p + ".attn.proj.weight"])
            do = torch.empty((M, D), dtype=torch.bfloat16, device=dev)
            ops.gemm_nn(gy, wp[p + ".attn.proj.weight"], do)
            dqkv = torch.empty((M, 3 * D), dtype=torch.bfloat16, device=dev)
            if self.variant == "v1":
                ops.attention_bwd(qkv.view(B, T, 3, self.H, self.hd), o.view(B, T, D), do.view(B, T, D), lse,
                                  dqkv.view(B, T, 3, self.H, self.hd), scale)
            else:
                tname = p + ".attn.relative_position_bias_table"
                tbl = sd[tname]
                ws, sh = self.windows[i]
                ops.attention2_bwd(qkv.view(B, T, 3, self.H, self.hd), o.view(B, T, D), do.view(B, T, D), lse,
                                   dqkv.view(B, T, 3, self.H, self.hd), scale, tbl, (tbl.shape[0] + 1) // 2, ws, sh,
                                   grads.get(tname), attn_drop, seed + 16 * i)
            side.run(ops.linear_wgrad, dqkv, h1, grads[p + ".attn.qkv.weight"])
            ops.colsum_bf16(dqkv, grads[p + ".attn.qkv.bias"])      # (uses the shared scratch: stays on this stream)
            dh1 = torch.empty((M, D), dtype=torch.bfloat16, device=dev)
            ops.gemm_nn(dqkv, wp[p + ".attn.qkv.weight"], dh1)
            ops.row_ln_bwd(dh1, x1, m1, r1s, sd[p + ".norm1.weight"], gx, True, grads[p + ".norm1.weight"],
                           grads[p + ".norm1.bias"])
        if on_stage is not None:
            side.join()
            on_stage("transformer")          # every blocks.* / norm / head gradient is final
        dtok = ops.tokens_bwd(gx, ctx.mask, grads["mask_token"].view(-1), B, T, D)
        g = ops.pool_bwd(dtok.view(B, 1, T, D), ctx.idx2, ctx.l3_shape)

        # ---- stem blocks ------------------------------------------------------------------------
        # conv weight gradients accumulate in the GEMM's natural output layout (split-K slices reduce-add in place) in
        # one zeroed buffer and are permuted into the OIHW .grad tensors by one launch per layout:
        #   "atoms": 3x3 convs with horizontal stride 1 - the two-accumulator, window-sharing GEMM,
        #            rows = (kernel row, 64-channel atom, kw): [3, Cin/64, 3, 64, Cout];
        #   "tco"  : other convs whose Cout is not a multiple of 128 - transposed GEMM, [taps, Cin, Cout];
        #   "ctc"  : the rest (stride-2 3x3, 1x1 downsamples of the 384 / 768-channel layers) - [Cout, taps, Cin]
        cnames = [k for k in wp if k.startswith("patch_embed.")]
        hstride = {}
        for (p, s, *_rest) in ctx.blocks:
            hstride[p + ".conv1.weight"] = s[1]
            hstride[p + ".conv2.weight"] = 1
        gt_flat = torch.zeros(sum(wp[k].numel() for k in cnames), dtype=torch.float32, device=dev)
        gt, layout, off = {}, {}, 0
        for k in cnames:
            co, tp, ci = wp[k].shape
            if tp == 9 and hstride.get(k, 0) == 1:
                layout[k], shape = "atoms", (3, ci // 64, 3, 64, co)
            elif co % 128:
                layout[k], shape = "tco", (tp, ci, co)
            else:
                layout[k], shape = "ctc", (co, tp, ci)
            gt[k] = gt_flat[off:off + wp[k].numel()].view(shape)
            off += wp[k].numel()

        def wgrad(dy, x, ks, sh, sw, name):
            side.run(wgrad_main, dy, x, ks, sh, sw, name)

        def wgrad_main(dy, x, ks, sh, sw, name):
            if layout[name] == "atoms":
                ops.conv_wgrad_acc_w(dy, x, sh, gt[name])
            elif layout[name] == "tco":
                ops.conv_wgrad_acc_t(dy, x, ks, sh, sw, gt[name])
            else:
                ops.conv_wgrad_acc(dy, x, ks, sh, sw, gt[name])
        unpacked = set()

        def unpack(pred):                # staged conv weight gradients -> the OIHW .grad tensors, one launch per layout
            sel = [k for k in cnames if k not in unpacked and pred(k)]
            unpacked.update(sel)
            side.join()                  # the staged gradients come from the side stream
            for lay, kw in (("atoms", dict(layout="atoms")), ("tco", dict(transposed=True)), ("ctc", dict())):
                part = [(gt[k], grads[k]) for k in sel if layout[k] == lay]
                if part:
                    ops.unpack_conv_grads(part, **kw)
        # [3][C] reduction targets of the 12 BatchNorm backward passes: one zeroed buffer per backward
        zs_total = sum(2 * 3 * blk[3].shape[-1] for blk in ctx.blocks)
        zs_pool, zs_off = torch.zeros(zs_total, dtype=torch.float32, device=dev), 0

        def zsum(C):
            nonlocal zs_off
            v = zs_pool[zs_off:zs_off + 3 * C]
            zs_off += 3 * C
            return v
        for (p, s, xin, r1, sa, a1, k1, r2, sb, rd, sdn, k2) in reversed(ctx.blocks):
            has_ds = rd is not None
            d2, dd, gz = ops.bn_bwd(
                g, k2, r2, sb, sd[p + ".bn2.weight"], grads[p + ".bn2.weight"], grads[p + ".bn2.bias"],
                raw_b=rd, st_b=sdn, gamma_b=sd[p + ".downsample.1.weight"] if has_ds else None,
                dgamma_b=grads[p + ".downsample.1.weight"] if has_ds else None,
                dbeta_b=grads[p + ".downsample.1.bias"] if has_ds else None, want_gz=not has_ds,
                zero_sums=zsum(r2.shape[-1]))
            wgrad(d2, a1, 3, 1, 1, p + ".conv2.weight")
            # conv2's input gradient with bn1's backward reduction in its epilogue (masked gradient + [2][C] sums), then
            # the apply pass alone; shapes the fused kernel does not serve take the two-pass route
            zs1 = zsum(r1.shape[-1])
            w2t = wp.get("T:" + p + ".conv2.weight")
            da1 = ops.conv_dgrad_bn(d2, w2t, tuple(a1.shape), r1, k1, sa, zs1) if (w2t is not None and FUSE_BN_BWD) else None
            if da1 is not None:
                d1 = ops.bn_bwd_apply(da1, r1, sa, sd[p + ".bn1.weight"], grads[p + ".bn1.weight"],
                                      grads[p + ".bn1.bias"], zs1)
            else:
                da1 = ops.conv_dgrad(d2, wp[p + ".conv2.weight"], tuple(a1.shape), 3, 1, 1, w_t=w2t)
                d1, _, _ = ops.bn_bwd(da1, k1, r1, sa, sd[p + ".bn1.weight"], grads[p + ".bn1.weight"],
                                      grads[p + ".bn1.bias"], zero_sums=zs1)
            wgrad(d1, xin, 3, s[0], s[1], p + ".conv1.weight")
            if has_ds:
                gin = ops.conv_dgrad(d1, wp[p + ".conv1.weight"], tuple(xin.shape), 3, s[0], s[1],
                                     w_t=wp.get("T:" + p + ".conv1.weight"))
                wgrad(dd, xin, 1, s[0], s[1], p + ".downsample.0.weight")
                ops.conv_dgrad(dd, wp[p + ".downsample.0.weight"], tuple(xin.shape), 1, s[0], s[1], dx=gin,
                               accumulate=True, w_t=wp.get("T:" + p + ".downsample.0.weight"))
            else:
                gin = ops.conv_dgrad(d1, wp[p + ".conv1.weight"], tuple(xin.shape), 3, s[0], s[1], dx=gz,
                                     accumulate=True, w_t=wp.get("T:" + p + ".conv1.weight"))
            g = gin
            if on_stage is not None and p == "patch_embed.%s.0" % STEM_LAYERS[-1][0]:
                # the last stem layer holds 3/4 of the stem's parameters: its gradients are final here, long before the
                # rest of the stem backward - unpack them now so that their all-reduce can start (data parallel)
                unpack(lambda k: k.startswith("patch_embed.%s." % STEM_LAYERS[-1][0]))
                on_stage("stem:" + STEM_LAYERS[-1][0])
        unpack(lambda k: k not in unpacked)
        # ---- stem head: pool -> relu -> bn1 -> conv1 ---------------------------------------------
        ops.stem_head_bwd(g, ctx.code1, ctx.x0, sd["patch_embed.conv1.weight"], ctx.moments,
                          sd["patch_embed.bn1.weight"], ctx.st1, grads["patch_embed.bn1.weight"],
                          grads["patch_embed.bn1.bias"], grads["patch_embed.conv1.weight"])
        self._wp_busy = max(0, getattr(self, "_wp_busy", 0) - 1)       # this forward's packed weights are free again
        return grads
