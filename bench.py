#!/usr/bin/env python
"""Benchmark of the HTR-VT hot path on B200 (driver contract: one JSON line on stdout from rank 0).

  python bench.py [--gpus N] [--steps K] [--warmup W]            our sm_100a path, training step (headline)
  python bench.py --workload infer [--gpus N] ...                batched inference + greedy CTC decode (config 4)
  python bench.py --impl reference ...                           the reference algorithm on the host CPU
  python bench.py ... --dump-outputs DIR                         also write what the last timed step returned as
                                                                 DIR/<name>.npy (same arguments -> same inputs)

Workload (BASELINE.json configs[1]): one HTR-VT IAM-shape training step = encoder forward (train mode,
span masking 0.4/8) + CTC loss + backward of every trainable parameter, batch 128 per GPU, 1x64x512
line images, 80 classes, bf16 tensor-core math with fp32 masters, driven through the reference's own call
sequence (model_v1/train.py:21-30: model(image, mask_ratio, max_span, use_masking=True) -> .float() ->
permute -> log_softmax -> criterion(...).mean() -> backward).  N > 1: batch sharding, NCCL gradient
all-reduce inside backward ("scaling": "weak").
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NB_CLS, IMG_H, IMG_W = 80, 64, 512
MASK_RATIO, MAX_SPAN = 0.4, 8
# algorithmic forward FLOPs per image (SURVEY.md 8d): stem 30.558 G + linears 7.263 G + attention 0.201 G
GFLOP_FWD_PER_IMG = 38.02


def synth_batch(B, seed):
    import numpy as np
    import torch
    rs = np.random.RandomState(seed)
    img = torch.from_numpy(rs.rand(B, 1, IMG_H, IMG_W).astype("float32"))
    lens = rs.randint(16, 65, size=B).astype("int32")
    tg = rs.randint(1, NB_CLS, size=int(lens.sum())).astype("int32")
    return img, torch.from_numpy(tg), torch.from_numpy(lens)


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe).  nvidia-smi needs
    0.1-0.5 s before its first sample, about as long as a 20-step timed region: the sampler is therefore started in
    front of the warm-up steps, every sample carries nvidia-smi's own wall-clock time stamp, and only the samples between
    mark() (timed region starts) and stop() are reported; if none fell inside (a very short region), the samples of
    the warm-up (same kernels, same load) are reported and `window` says so."""

    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.path = tempfile.mktemp(prefix="htrvt_clocks_", suffix=".csv")
        self.proc = None
        self.t0 = None

    def start(self):
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=self.fh,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
            return
        t_end = time.time() + 3.0                  # nvidia-smi's first sample: the loop is running from here on
        while time.time() < t_end:
            try:
                self.fh.flush()
                if os.path.getsize(self.path) > 0:
                    break
            except Exception:
                break
            time.sleep(0.02)

    def mark(self):
        self.t0 = time.time()

    def stop(self):
        import datetime
        t1 = time.time()
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.fh.close()
        rows = []
        try:
            for line in open(self.path):
                f = [v.strip() for v in line.split(",")]
                if len(f) < 10:
                    continue
                try:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                except Exception:
                    ts = None
                rows.append((ts, float(f[2]), float(f[3]),
                             [name for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                                       "sw_power_cap"), f[6:10]) if v.lower().startswith("active")]))
            os.unlink(self.path)
        except Exception:
            pass
        inside = [r for r in rows if self.t0 is not None and r[0] is not None and self.t0 <= r[0] <= t1]
        window = "timed region"
        if not inside:
            inside, window = rows, "warm-up + timed region (no sample fell inside the timed region)"
        if inside:
            sm = sorted(r[1] for r in inside)
            reasons = set()
            for r in inside:
                reasons.update(r[3])
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(r[2] for r in inside), reasons=sorted(reasons),
                       samples=len(inside), window=window)
        return out


def cpu_reference_rate(steps, warmup, B=8, seed=0):
    """The reference algorithm (CPU oracle port of model_v1 forward/backward + nn.CTCLoss) on the host cores,
    on a bounded sample of the workload: B images per step.  Returns (img/s, seconds per step, threads)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import htrvt_oracle as O
    # all the host threads this process may use: torchrun exports OMP_NUM_THREADS=1 to every rank, which would
    # quietly turn the multi-threaded CPU arm into a single-threaded one
    try:
        ncpu = len(os.sched_getaffinity(0))
    except AttributeError:
        ncpu = os.cpu_count() or 1
    if torch.get_num_threads() < ncpu:
        torch.set_num_threads(ncpu)
    torch.manual_seed(123)
    sd = O.init_state_dict(NB_CLS, [IMG_H, IMG_W], seed=123)
    img, tg, tl = synth_batch(B, seed)
    times = []
    for i in range(warmup + steps):
        mask = O.draw_span_mask(IMG_W // 4, MASK_RATIO, MAX_SPAN)
        t0 = time.perf_counter()
        O.train_step(sd, img, tg, tl, mask)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    per = sum(times) / len(times)
    return B / per, per, torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B = 8
    if args.workload == "infer":
        rate, per, threads = cpu_reference_infer_rate(args.steps, max(args.warmup, 1), B=B)
        print(json.dumps({
            "impl": "reference", "metric": "line images/sec (inference)", "value": rate, "unit": "img/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "v1_infer_greedy_decode_512_lines_per_gpu_64x512_c80",
                       "sample": "%d lines per step on the host CPU" % B},
            "cpu_baseline": {"value": rate, "unit": "img/s", "cores": threads, "kind": "port",
                             "sample": "oracle port of model_v1 eval forward + reference decode, %d lines/step, %d steps"
                                       % (B, args.steps)},
            "e2e": {"value": rate, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)
        return
    rate, per, threads = cpu_reference_rate(args.steps, max(args.warmup, 1), B=B)
    line = {
        "impl": "reference", "metric": "line images/sec (train step)", "value": rate, "unit": "img/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "v1_train_step_b128_64x512_c80", "sample": "%d images per step on the host CPU" % B},
        "cpu_baseline": {"value": rate, "unit": "img/s", "cores": threads, "kind": "port",
                         "sample": "oracle port of model_v1 fwd+bwd+CTCLoss, %d images/step, %d steps" % (B, args.steps)},
        "e2e": {"value": rate, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def inference_metrics(torch, dist, dev, h, ops, model, world, rank, steps, lines_per_gpu=512, keep=None):
    """BASELINE.json config 4: batched inference + greedy CTC decode, 512 synthetic lines per GPU (4096 over 8 GPUs),
    sharded by batch with NO collective on the data path (ddp.shard_batch); each rank decodes its own shard to Python
    strings.  Two timings, both max over ranks between barriers:
      value : images resident in HBM, eval forward + decode kernels (ids stay on the device);
      e2e   : through the public API with HOST buffers - pinned fp32 images -> H2D -> model(image) ->
              converter.decode_logits (argmax + collapse on device, ONE D2H copy of ids + lengths, id -> str).
    keep: a dict that receives the logits, ids and lengths of the last resident batch."""
    conv = h.CTCLabelConverter("".join(chr(33 + i) for i in range(NB_CLS - 1)))
    img_h = synth_batch(lines_per_gpu, 1000 + rank)[0].pin_memory()
    img_d = img_h.to(dev)
    was_training = model.training
    model.eval()

    def resident():
        with torch.no_grad():
            logits = model(img_d).float()
            ids, lens = h.greedy_decode(logits, NB_CLS)
        if keep is not None:
            keep.update(logits=logits, ids=ids, lens=lens)
        return ids, lens

    pf = h.HostPrefetcher(dev)                   # batch i+1's 67 MB H2D copy runs under batch i's kernels
    pf.put(img_h)

    pending = [None]

    def e2e():
        # one batch in flight behind the host: the strings of batch i - 1 are built (after ITS ids arrived in pinned
        # memory) while batch i's kernels run; every batch's ids are read back inside the timed region (drain below)
        with torch.no_grad():
            image = pf.get()
            pf.put(img_h)
            cur = conv.decode_logits_async(model(image).float())
        out = pending[0].strings() if pending[0] is not None else None
        pending[0] = cur
        return out

    def drain():
        out = pending[0].strings() if pending[0] is not None else None
        pending[0] = None
        return out

    def timed(fn, iters, drain=None):
        for _ in range(3):
            fn()
        if drain is not None:
            drain()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        if drain is not None:
            drain()                       # the last batch's strings, still inside the timed region
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / iters], device=dev)
        if world > 1:
            dist.barrier()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    n0 = ops.launch_count()
    ms = timed(resident, steps)
    launches = (ops.launch_count() - n0) // (steps + 3)
    ms_e2e = timed(e2e, steps, drain)
    e2e()
    strings = drain()
    T = IMG_W // 4
    if was_training:
        model.train()
    return {"img_per_s": world * lines_per_gpu / (ms * 1e-3), "ms_per_batch": ms, "lines_per_gpu": lines_per_gpu,
            "n_gpus": world, "gpu_launches_per_batch": launches,
            "e2e": {"value": world * lines_per_gpu / (ms_e2e * 1e-3), "unit": "img/s", "ms_per_batch": ms_e2e,
                    "h2d_bytes_per_step": img_h.numel() * 4, "d2h_bytes_per_step": lines_per_gpu * (T + 1) * 4,
                    "pipelining": "HostPrefetcher (H2D of batch i+1 under batch i) + decode_logits_async (strings of "
                                  "batch i-1 built on the host under batch i's kernels; every batch read back inside "
                                  "the timed region)"},
            "decoded_lines": len(strings), "collective": "none (batch sharding; strings stay on their rank)",
            "what": "eval-mode forward + greedy CTC decode (BASELINE config 4: 512 lines per GPU)"}


def gpu_eager_baseline(torch, dev, B=128, steps=3):
    """GPU-side baseline on the SAME box: the reference's graph (the oracle's functional restatement of
    model_v1/model/HTR_VT.py + resnet18.py, pinned to the reference by tests/test_oracle.py) run by torch eager with the
    stock library kernels - cuDNN convolutions, cuBLAS GEMMs, ATen LayerNorm / softmax / native CTC ("the existing
    Blackwell path").  None of this repo's kernels run here; it is a reported baseline like cpu_baseline, ~10 s."""
    import torch.nn.functional as F
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import htrvt_oracle as O
    sd0 = O.init_state_dict(NB_CLS, [IMG_H, IMG_W], seed=123)
    img, tg, tl = synth_batch(B, 0)
    img, tg_d, tl_d = img.to(dev), tg.to(dev), tl.to(dev)
    T = IMG_W // 4
    mask = O.draw_span_mask(T, MASK_RATIO, MAX_SPAN).to(dev)
    in_len = torch.full((B,), T, dtype=torch.int32, device=dev)
    out = {}
    for mode, autocast in (("fp32", False), ("bf16_autocast", True)):
        sd = {k: v.to(dev) for k, v in sd0.items()}
        for k, v in sd.items():
            if v.is_floating_point() and "running_" not in k and k != "pos_embed":
                sd[k] = v.clone().requires_grad_(True)

        def step():
            for v in sd.values():
                if v.requires_grad:
                    v.grad = None
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                logits = O.forward(sd, img, mask=mask, training=True)
            lp = logits.float().permute(1, 0, 2).log_softmax(2)
            prev = torch.backends.cudnn.enabled
            torch.backends.cudnn.enabled = False                     # model_v1/train.py:26
            loss = F.ctc_loss(lp, tg_d, in_len, tl_d, blank=0, reduction="none", zero_infinity=True).mean()
            torch.backends.cudnn.enabled = prev
            loss.backward()

        for _ in range(3):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[mode] = {"train_step_ms": ms, "img_per_s": B / (ms * 1e-3)}
        del sd
        torch.cuda.empty_cache()
    out["what"] = ("the reference graph (oracle restatement) through torch %s eager on this GPU: cuDNN / cuBLAS / ATen "
                   "CTC, batch %d; fp32 = the reference's own arithmetic (TF32 convs as torch defaults), bf16 = autocast"
                   % (torch.__version__, B))
    return out


def extra_metrics(torch, dev, h, ops, H, model, peaks):
    """The other BASELINE.json metrics / configs, measured on the same box right after the headline run (1 GPU):
    CTC loss+grad us/batch with its HBM roofline fraction, inference (eval forward + greedy decode) img/s at the
    per-GPU share of config 4 (512 lines), and the windowed wide-line variant's training step (config 5)."""
    from importlib import import_module
    out = {}
    hbm = float(peaks.get("hbm_gbs", 6500.0))

    def timed_ms(fn, iters, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    def timed_graph_ms(fn, iters):
        """Per-call GPU time of a tiny kernel: `iters` calls captured into ONE CUDA graph and replayed, so the number
        is the kernels' back-to-back time and not the host's enqueue rate (the ctypes + torch.empty path costs more
        than a 5-10 us kernel)."""
        fn()
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            fn()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                for _ in range(iters):
                    fn()
        torch.cuda.current_stream().wait_stream(side)
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / (3 * iters)

    # ---- CTC loss + gradient, B=128, T=128, C=80, fused log-softmax (one launch); 16 rotating buffers (168 MB of
    # logits + gradients > 126 MB L2) so no iteration finds its data in L2
    B, T, C = 128, 128, NB_CLS
    g = torch.Generator(device="cpu").manual_seed(0)
    bufs = [torch.randn(B, T, C, generator=g).to(dev) for _ in range(16)]
    _, tg, tl = synth_batch(B, 0)
    tg, tl_d = tg.to(dev), tl.to(dev)
    mtl = int(tl.max())
    state = {"i": 0}

    def ctc_once():
        x = bufs[state["i"] % len(bufs)]
        state["i"] += 1
        ops.ctc_loss_grad(x, tg, None, tl_d, layout="btc", is_logprob=False, want_grad=True, max_target_len=mtl,
                          grad_scale_const=1.0 / B)

    ms = timed_ms(ctc_once, 64)
    bytes_ctc = 2.0 * B * T * C * 4 + float(tg.numel()) * 4 + 12.0 * B
    out["ctc_loss_grad"] = {"us_per_batch": ms * 1e3, "batch": B, "T": T, "C": C, "algorithmic_bytes": bytes_ctc,
                            "achieved_gbs": bytes_ctc / (ms * 1e-3) / 1e9, "hbm_peak_gbs": hbm,
                            "frac_of_hbm_roofline": bytes_ctc / (ms * 1e-3) / 1e9 / hbm,
                            "note": "T sequential alpha/beta steps bound this kernel by latency, not bytes; the "
                                    "recursion runs in the linear domain on the FP64 pipe (fallbacks to log space: %d)"
                                    % ops.lib().htrvt_ctc_fallback_count()}
    del bufs
    # a batch that fills the chip: the lane-group throughput kernel (ctc_grp.cu, automatic for B >= 1024)
    Bl = 4096
    xl = torch.randn(Bl, T, C, device=dev)
    _, tgl, tll = synth_batch(Bl, 3)
    tgl, tll_d, mtl_l = tgl.to(dev), tll.to(dev), int(tll.max())
    ms = timed_ms(lambda: ops.ctc_loss_grad(xl, tgl, None, tll_d, layout="btc", is_logprob=False, want_grad=True,
                                            max_target_len=mtl_l, grad_scale_const=1.0 / Bl), 10)
    bl = 2.0 * Bl * T * C * 4 + float(tgl.numel()) * 4 + 12.0 * Bl
    out["ctc_loss_grad"]["batch_4096"] = {"us_per_batch": ms * 1e3, "achieved_gbs": bl / (ms * 1e-3) / 1e9,
                                          "frac_of_hbm_roofline": bl / (ms * 1e-3) / 1e9 / hbm,
                                          "kernel": "ctc_grp_kernel<8, 3> (8 lanes per sequence, fp32 linear domain) + "
                                                    "fix-up launch",
                                          "flagged_for_fixup": int(ops.lib().htrvt_ctc_flagged_count())}
    del xl
    # the wide-line shape (BASELINE config 5): T = 256, C = 90, labels 64..200 -> up to 401 states per sequence
    try:
        import numpy as np
        Bw, Tw, Cw = 128, 256, 90
        xw = torch.randn(Bw, Tw, Cw, device=dev)
        rsw = np.random.RandomState(5)
        lw = rsw.randint(64, 201, size=Bw).astype("int32")
        tgw = torch.from_numpy(rsw.randint(1, Cw, size=int(lw.sum())).astype("int32")).to(dev)
        tlw = torch.from_numpy(lw).to(dev)
        ms = timed_ms(lambda: ops.ctc_loss_grad(xw, tgw, None, tlw, layout="btc", is_logprob=False, want_grad=True,
                                                max_target_len=int(lw.max()), grad_scale_const=1.0 / Bw), 20)
        bw = 2.0 * Bw * Tw * Cw * 4 + float(tgw.numel()) * 4 + 12.0 * Bw
        out["ctc_loss_grad"]["wide_T256_C90_L200"] = {"us_per_batch": ms * 1e3, "batch": Bw,
                                                      "achieved_gbs": bw / (ms * 1e-3) / 1e9,
                                                      "frac_of_hbm_roofline": bw / (ms * 1e-3) / 1e9 / hbm}
        del xw
    except Exception as e:
        out["ctc_loss_grad"]["wide_T256_C90_L200"] = {"error": repr(e)[:200]}

    # ---- greedy decode kernel alone (argmax + collapse): 512 lines x 128 frames x 80 classes of fp32 logits; 8
    # rotating buffers (168 MB > 126 MB L2) so every call streams from HBM
    try:
        Bd, Td = 512, IMG_W // 4
        dbufs = [torch.randn(Bd, Td, NB_CLS, device=dev) for _ in range(8)]
        dstate = {"i": 0}

        def dec_once():
            x = dbufs[dstate["i"] % len(dbufs)]
            dstate["i"] += 1
            ops.greedy_decode_ids(x, NB_CLS)

        ms_host = timed_ms(dec_once, 64)
        try:
            ms = timed_graph_ms(dec_once, 64)
        except Exception:
            ms = ms_host
        bytes_dec = Bd * Td * NB_CLS * 4.0 + Bd * Td * 4.0 + Bd * 4.0
        out["greedy_decode"] = {"us_per_batch": ms * 1e3, "us_per_call_host_enqueued": ms_host * 1e3,
                                "timing": "64 calls in one CUDA graph (kernel time, not host enqueue rate)",
                                "lines": Bd, "T": Td, "C": NB_CLS,
                                "algorithmic_bytes": bytes_dec, "achieved_gbs": bytes_dec / (ms * 1e-3) / 1e9,
                                "hbm_peak_gbs": hbm, "frac_of_hbm_roofline": bytes_dec / (ms * 1e-3) / 1e9 / hbm}
        del dbufs
    except Exception as e:
        out["greedy_decode"] = {"error": repr(e)[:200]}

    # ---- inference: eval forward + greedy decode (argmax + collapse on device, one D2H copy), 512 lines per GPU
    Bi = 512
    conv = h.CTCLabelConverter("".join(chr(33 + i) for i in range(NB_CLS - 1)))
    img = synth_batch(Bi, 1)[0].to(dev)
    model.eval()

    def infer_once():
        with torch.no_grad():
            preds = model(img)
            return conv.decode_logits(preds.float())

    infer_once()
    # validation metrics on device (SURVEY.md 8f row 3): Levenshtein of the decoded ids against the label ids
    try:
        with torch.no_grad():
            preds = model(img).float()
        ids, lens = h.greedy_decode(preds, NB_CLS)
        _, tgv, tlv = synth_batch(Bi, 4)
        tgv = tgv.to(dev)
        ms_ed = timed_ms(lambda: h.cer_from_ids(ids, lens, tgv, tlv), 20)
        out["cer_device"] = {"us_per_batch": ms_ed * 1e3, "pairs": Bi,
                             "what": "edit distances of 512 decoded id rows vs label ids, one launch (valid.py:49-55)"}
    except Exception as e:
        out["cer_device"] = {"error": repr(e)[:200]}
    # ---- LM-rescoring evaluation (model_window/test_with_kenlm.py:25-59): K-best paths of 512 lines in one launch +
    # one D2H copy + the host-side string building / scorer calls, against the reference's per-frame Python beam
    try:
        class _LenLM(object):
            def score(self, text):
                return -0.1 * len(text)

        lp = torch.randn(IMG_W // 4, Bi, NB_CLS, device=dev).log_softmax(2)
        ms_k = timed_ms(lambda: ops.ctc_kbest_paths(lp, 5), 20)
        ms_b = timed_ms(lambda: h.beam_search_with_lm_batch(lp, conv, _LenLM(), beam_size=5), 3, warm=1)
        out["kbest_beam"] = {"kernel_us_per_batch": ms_k * 1e3, "with_host_strings_ms_per_batch": ms_b, "lines": Bi,
                             "beam": 5, "what": "K-best CTC paths on device + LM pick on host (test_with_kenlm.py:25-59)"}
        # the true prefix beam search (SURVEY.md 8(f) row 4): labellings instead of alignment paths
        out["prefix_beam"] = {}
        for Kb in (5, 16):
            ms_p = timed_ms(lambda: ops.ctc_prefix_beam(lp, Kb), 10)
            out["prefix_beam"]["beam_%d_us_per_batch" % Kb] = ms_p * 1e3
        ms_pb = timed_ms(lambda: h.beam_search_with_lm_batch(lp, conv, _LenLM(), beam_size=5, search="prefix"), 3, warm=1)
        out["prefix_beam"].update({"with_host_strings_ms_per_batch_beam_5": ms_pb, "lines": Bi, "T": IMG_W // 4,
                                   "C": NB_CLS, "what": "CTC prefix beam search, one warp per line, all classes "
                                   "extended every frame, float64 log-space scores (csrc/prefix_beam.cu)"})
        del lp
    except Exception as e:
        out["kbest_beam"] = {"error": repr(e)[:200]}
    # ---- training-time augmentation (SURVEY.md 8(f) row 2; dataset.py:13-45): all three stages on 128 uint8 lines
    try:
        import types
        import numpy as np
        aug = import_module("htr-vt_b200.augment")
        a_args = types.SimpleNamespace(proj=8.0, dila_ero_max_kernel=3, dila_ero_iter=1, jitter_contrast=0.4,
                                       jitter_brightness=0.4, jitter_saturation=0.4, jitter_hue=0.2)
        st_np, st_t = np.random.get_state(), torch.random.get_rng_state()
        xa = torch.randint(0, 256, (128, IMG_H, IMG_W), dtype=torch.uint8, device=dev)
        seed = 0
        while True:
            seed += 1
            np.random.seed(seed); torch.manual_seed(seed)
            pa = aug.draw_collate_params(128, IMG_H, IMG_W, a_args)
            if all(pa[k] is not None for k in ("warp", "morph", "jitter")):
                break
        t0 = time.perf_counter()
        for _ in range(5):
            np.random.seed(seed); torch.manual_seed(seed)
            aug.draw_collate_params(128, IMG_H, IMG_W, a_args)
            rec, morph = aug.pack_params(pa, 128, IMG_H, IMG_W)
        host_ms = (time.perf_counter() - t0) / 5 * 1e3
        recd = torch.from_numpy(rec).to(dev)
        ms_a = timed_ms(lambda: ops.augment_lines(xa, recd, morph), 20)
        np.random.set_state(st_np); torch.random.set_rng_state(st_t)
        out["augment"] = {"kernel_us_per_batch": ms_a * 1e3, "host_draws_and_records_ms_per_batch": host_ms,
                          "lines": 128, "img": [IMG_H, IMG_W],
                          "what": "SameTrCollate's projective warp + resize, erosion / dilation and brightness / "
                                  "contrast jitter on 128 uint8 lines in one launch; random decisions drawn on the "
                                  "host in the reference's order (dataset.py:13-45 runs PIL / OpenCV / scikit-image "
                                  "per image)"}
        del xa
    except Exception as e:
        out["augment"] = {"error": repr(e)[:200]}
    model.train()
    del img

    # ---- training step fed with the loader's uint8 lines (SURVEY.md 8f row 2): 4x fewer PCIe bytes, conversion +
    # padding + input LayerNorm in one kernel; same timed region as the headline e2e (H2D + step + loss.item())
    try:
        import numpy as np
        Bu = 128
        u8_h = torch.from_numpy(np.random.RandomState(6).randint(0, 256, size=(Bu, 1, IMG_H, IMG_W)).astype("uint8")).pin_memory()
        _, tgu, tlu = synth_batch(Bu, 6)
        tgu, tlu = tgu.pin_memory(), tlu.pin_memory()
        uparams = [p for p in model.parameters() if p.requires_grad]

        def step_u8():
            for p in uparams:
                p.grad = None
            preds = model(u8_h.to(dev, non_blocking=True), MASK_RATIO, MAX_SPAN, use_masking=True)
            loss = h.ctc_loss_from_logits(preds.float(), tgu.to(dev, non_blocking=True), tlu).mean()
            loss.backward()
            return loss.item()

        ms = timed_ms(step_u8, 5, warm=2)
        out["e2e_uint8_input"] = {"img_per_s": Bu / (ms * 1e-3), "ms_per_step": ms,
                                  "h2d_bytes_per_step": u8_h.numel() + tgu.numel() * 4,
                                  "what": "train step from pinned uint8 line images through model.forward(uint8)"}
        for p in uparams:
            p.grad = None
    except Exception as e:
        out["e2e_uint8_input"] = {"error": repr(e)[:200]}

    # ---- the reference's full training iteration (model_v1/train.py:113-126): SAM(AdamW) = two forward/backward
    # passes around first_step / second_step + the EMA update, with the multi-tensor optimizer kernels
    try:
        SAMm = import_module("htr-vt_b200.utils.sam")
        Um = import_module("htr-vt_b200.utils.utils")
        Bs = 128
        imgs, tgs, tls = [t.to(dev) for t in synth_batch(Bs, 2)]
        opt = SAMm.SAM(model.parameters(), torch.optim.AdamW, lr=1e-4, betas=(0.9, 0.99), weight_decay=0.5)
        ema = Um.ModelEma(model, 0.9999)
        crit = h.CTCLoss(reduction="none", zero_infinity=True)
        ps = torch.full((Bs,), IMG_W // 4, dtype=torch.int32, device=dev)

        def fb():
            preds = model(imgs, MASK_RATIO, MAX_SPAN, use_masking=True).float()
            loss = crit(preds.permute(1, 0, 2).log_softmax(2), tgs, ps, tls).mean()
            loss.backward()

        def sam_iter():
            opt.zero_grad()
            fb()
            opt.first_step(zero_grad=True)
            fb()
            opt.second_step(zero_grad=True)
            model.zero_grad()
            ema.update(model, num_updates=10)

        def opt_only():
            for p in model.parameters():
                if p.requires_grad and p.grad is None:
                    p.grad = torch.zeros_like(p)
            opt.first_step(zero_grad=False)
            opt.second_step(zero_grad=False)
            ema.update(model, num_updates=10)

        def opt_device_ms(reps=5):
            """Device time of the optimizer launches alone: a forward/backward (~17 ms of queued kernels) goes first so
            that the host has finished enqueueing first_step / second_step / EMA long before the device reaches them -
            the event pair then brackets the kernels back to back, not the ~2 ms of Python that builds the pointer
            tables of 101 tensors (which, in a real iteration, runs under the previous pass's kernels)."""
            ts = []
            for _ in range(reps):
                opt.zero_grad()
                fb()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                opt_only()
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            return sorted(ts)[len(ts) // 2]

        ms = timed_ms(sam_iter, 5, warm=2)
        ms_opt = timed_ms(opt_only, 5, warm=1)
        ms_opt_dev = opt_device_ms()
        nparam = sum(p.numel() for p in model.parameters() if p.requires_grad)
        # norm: g (4); climb: p, g -> old, p (16); restore + AdamW: old, g, m, v -> m, v, p (28); EMA: ema, src -> ema (12)
        opt_bytes = nparam * (4 + 16 + 28 + 12)
        opt_gbs = opt_bytes / (ms_opt_dev * 1e-3) / 1e9
        out["sam_iteration"] = {"img_per_s": Bs / (ms * 1e-3), "ms_per_iteration": ms, "batch_per_gpu": Bs,
                                "optimizer_ms": ms_opt_dev, "optimizer_algorithmic_bytes": opt_bytes,
                                "optimizer_gbs": opt_gbs, "hbm_peak_gbs": hbm,
                                "optimizer_frac_of_hbm_roofline": opt_gbs / hbm,
                                "optimizer_ms_host_bound": ms_opt,
                                "optimizer_timing": "optimizer_ms: CUDA events around the 4 multi-tensor passes with "
                                                    "the host enqueued ahead (behind a forward/backward); "
                                                    "optimizer_ms_host_bound: the same calls on an idle stream, "
                                                    "where the Python that builds the pointer tables is the limit",
                                "what": "2x(fwd+bwd+CTC) + SAM first/second step (fused AdamW) + EMA, train.py:113-126"}
        del opt, ema
        for p in model.parameters():
            p.grad = None
    except Exception as e:
        out["sam_iteration"] = {"error": repr(e)[:200]}

    # ---- windowed variant (model_window), 64x1024 lines, T = 256, 90 classes, labels up to 200: training step with
    # the reference's train-mode regularisers on (dropout 0.1 / attention dropout 0.05 / DropPath <= 0.1)
    try:
        Wm = import_module("htr-vt_b200.model_window.HTR_VT")
        import numpy as np
        Bw, Ww, Cw = 128, 1024, 90
        torch.manual_seed(123)
        wm = Wm.create_model(Cw, [IMG_H, Ww]).to(dev).train()
        rs = np.random.RandomState(5)
        imgw = torch.from_numpy(rs.rand(Bw, 1, IMG_H, Ww).astype("float32")).to(dev)
        lens = rs.randint(64, 201, size=Bw).astype("int32")
        tgw = torch.from_numpy(rs.randint(1, Cw, size=int(lens.sum())).astype("int32")).to(dev)
        tlw = torch.from_numpy(lens)
        wparams = [p for p in wm.parameters() if p.requires_grad]

        def win_step():
            for p in wparams:
                p.grad = None
            preds = wm(imgw, MASK_RATIO, MAX_SPAN, use_masking=True)
            loss = h.ctc_loss_from_logits(preds.float(), tgw, tlw).mean()
            loss.backward()

        ms = timed_ms(win_step, 3, warm=2)
        out["window_train_step"] = {"img_per_s": Bw / (ms * 1e-3), "ms_per_step": ms, "batch_per_gpu": Bw,
                                    "img": [1, IMG_H, Ww], "nb_cls": Cw, "T": Ww // 4,
                                    "what": "model_window fwd+bwd+CTC (BASELINE config 5)"}
        del wm, imgw
    except Exception as e:                                   # never lose the headline line to an extra
        out["window_train_step"] = {"error": repr(e)[:200]}
    torch.cuda.empty_cache()
    return out


def setup_ours():
    """One process per GPU (RANK / LOCAL_RANK / WORLD_SIZE from torchrun), NCCL up, package imported."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the hot path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL writes its version banner / debug lines to stdout while the communicator comes up; rank 0's stdout must
        # carry ONE JSON line, so file descriptor 1 points at stderr until the first collective has completed
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    from importlib import import_module
    import __graft_entry__ as ge
    ge.ensure_built()
    import htrvt_b200 as h
    ops = import_module("htr-vt_b200.ops")
    H = import_module("htr-vt_b200.model.HTR_VT")
    return torch, dist, world, rank, local, dev, h, ops, H


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    return json.load(open(p)) if os.path.exists(p) else {}


DUMP_LIMIT_BYTES = 64 * 10 ** 6
GRAD_SAMPLE = 1 << 22              # gradient entries --dump-outputs writes (16.8 MB of the 214 MB of one step)


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each array as out_dir/<name>.npy.  float64 stays float64, other floating point becomes float32,
    integers (token ids, lengths) become float64, which holds them exactly."""
    import numpy as np
    out = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        out[name] = a if a.dtype == np.float64 else a.astype(np.float64 if a.dtype.kind in "iub" else np.float32)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("bench.py: --dump-outputs would write %d bytes (limit %d)" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def train_step_outputs(torch, loss, logits, params):
    """What one training step hands its caller: the loss, the model's logits and every parameter's .grad.  The
    gradients are written as their per-tensor L2 norms (all tensors) and the entries at a fixed, seeded sample of
    positions in their concatenation (model.parameters() order, ascending positions)."""
    import numpy as np
    flat = torch.cat([p.grad.reshape(-1) for p in params])
    idx = np.sort(np.random.default_rng(0).choice(flat.numel(), min(GRAD_SAMPLE, flat.numel()), replace=False))
    return {"loss": loss, "logits": logits,
            "grad_norms": torch.stack([p.grad.double().norm() for p in params]),
            "grad_sample": flat[torch.from_numpy(idx).to(flat.device)]}


def run_infer(args):
    """--workload infer: BASELINE.json config 4 as its own JSON line (batched inference + greedy CTC decode, 512
    lines per GPU, batch sharding, no collective)."""
    torch, dist, world, rank, local, dev, h, ops, H = setup_ours()
    torch.manual_seed(123)
    model = H.create_model(NB_CLS, [IMG_H, IMG_W]).to(dev).eval()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    clocks.mark()                         # (inference_metrics warms up inside; its two timed legs follow back to back)
    last = {}
    m = inference_metrics(torch, dist, dev, h, ops, model, world, rank, steps=args.steps, keep=last)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    # roofline of the tap-GEMM family inside one inference batch (CUDA events per op on the launching stream)
    img = synth_batch(m["lines_per_gpu"], 1000 + rank)[0].to(dev)
    ops.PROFILE = []
    with torch.no_grad():
        h.greedy_decode(model(img).float(), NB_CLS)
    torch.cuda.synchronize()
    prof, ops.PROFILE = ops.PROFILE, None
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = load_peaks()
    g_ms = sum(a.elapsed_time(b) for n, fl, a, b in prof if n in ("gemm_tn", "conv_fwd"))
    g_fl = sum(fl for n, fl, a, b in prof if n in ("gemm_tn", "conv_fwd"))
    all_ms = sum(a.elapsed_time(b) for n, fl, a, b in prof)
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    ach = g_fl / (g_ms * 1e-3) / 1e12 if g_ms else 0.0
    by = {}
    for n, fl, a, b in prof:
        by[n] = by.get(n, 0.0) + a.elapsed_time(b)
    line = {"metric": "line images/sec (inference)", "value": m["img_per_s"], "unit": "img/s", "n_gpus": world,
            "steps": args.steps, "warmup": 3, "ms_per_step": m["ms_per_batch"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "v1_infer_greedy_decode_512_lines_per_gpu_64x512_c80", "lines_per_gpu": m["lines_per_gpu"],
                       "img": [1, IMG_H, IMG_W], "nb_cls": NB_CLS, "parallelism": "dp%d (batch sharding, no collective)" % world,
                       "l2": "one batch's activations (~1.5 GB) >> 126 MB L2; no flush needed",
                       "algorithmic_tflop_per_step": GFLOP_FWD_PER_IMG * m["lines_per_gpu"] / 1e3},
            "clocks": clk, "e2e": m["e2e"], "gpu_launches": m["gpu_launches_per_batch"] * args.steps,
            "roofline": {"bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": ach / peak_tf if peak_tf else None, "traffic": None,
                         "kernel": "tapgemm_kernel (conv / linear forward launches of one inference batch)",
                         "ms_in_step": g_ms, "share_of_step": g_ms / all_ms if all_ms else None,
                         "peak_source": "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback"},
            "breakdown_ms": {k: round(v, 3) for k, v in sorted(by.items(), key=lambda kv: -kv[1])}}
    if world == 1 and not args.no_cpu_baseline:
        rate, per, threads = cpu_reference_infer_rate(5, 1)
        line["cpu_baseline"] = {"value": rate, "unit": "img/s", "cores": threads, "kind": "port",
                                "sample": "oracle port of model_v1 eval forward + reference decode, 8 lines/step, 5 steps"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def cpu_reference_infer_rate(steps, warmup, B=8, seed=0):
    """Reference inference on the host cores: eval forward (oracle port) + log_softmax / max / decode as valid.py:31-42."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import htrvt_oracle as O
    try:
        ncpu = len(os.sched_getaffinity(0))
    except AttributeError:
        ncpu = os.cpu_count() or 1
    if torch.get_num_threads() < ncpu:
        torch.set_num_threads(ncpu)
    sd = O.init_state_dict(NB_CLS, [IMG_H, IMG_W], seed=123)
    img = synth_batch(B, seed)[0]
    alphabet = "".join(chr(33 + i) for i in range(NB_CLS - 1))
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        with torch.no_grad():
            lg = O.forward(sd, img, training=False)
        idx = O.argmax_first(lg.numpy()).reshape(-1)
        O.decode_strings(idx, [lg.shape[1]] * B, alphabet)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    per = sum(times) / len(times)
    return B / per, per, torch.get_num_threads()


def run_ours(args):
    torch, dist, world, rank, local, dev, h, ops, H = setup_ours()

    B = args.batch
    torch.manual_seed(123)
    model = H.create_model(NB_CLS, [IMG_H, IMG_W]).to(dev).train()
    if world > 1:
        model.enable_data_parallel()
    criterion = h.CTCLoss(reduction="none", zero_infinity=True).to(dev)
    img_h, tg_h, tl_h = synth_batch(B, seed=rank)
    img_h, tg_h, tl_h = img_h.pin_memory(), tg_h.pin_memory(), tl_h.pin_memory()
    img_d, tg_d, tl_d = img_h.to(dev), tg_h.to(dev), tl_h.to(dev)
    params = [p for p in model.parameters() if p.requires_grad]
    last = {}                                    # the latest step's logits and loss (--dump-outputs)

    def compute_loss(image, text, length):
        # model_v1/train.py:21-30 with the drop-in model / criterion
        preds = model(image, MASK_RATIO, MAX_SPAN, use_masking=True)
        preds = preds.float()
        last["logits"] = preds.detach()
        preds_size = torch.full((B,), preds.size(1), dtype=torch.int32, device=dev)
        preds = preds.permute(1, 0, 2).log_softmax(2)
        return criterion(preds, text, preds_size, length).mean()

    def step_resident():
        for p in params:
            p.grad = None
        loss = compute_loss(img_d, tg_d, tl_d)
        loss.backward()
        last["loss"] = loss
        return loss

    # end to end: every step copies ITS inputs from pinned host memory (16.8 MB) and reads its loss back.  The copies
    # go through the package's HostPrefetcher: the batch of step i+1 is copied on a side stream while step i computes
    # (what a DataLoader-fed train.py does with `pf.put(next_batch)`); one copy per step, inside the timed region.
    pf = h.HostPrefetcher(dev)
    pf.put(img_h, tg_h, tl_h)

    def step_e2e_sync():
        for p in params:
            p.grad = None
        image, text, length = pf.get()
        pf.put(img_h, tg_h, tl_h)                # the next step's inputs
        loss = compute_loss(image, text, length)
        loss.backward()
        return loss.item()                       # train.py:129 as written: a device sync every step

    meter = h.RunningLoss()

    def step_e2e():
        for p in params:
            p.grad = None
        image, text, length = pf.get()
        pf.put(img_h, tg_h, tl_h)                # the next step's inputs
        loss = compute_loss(image, text, length)
        loss.backward()
        meter.add(loss)                          # D2H read of the step's result, every step, without stalling the host

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, drain=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if drain is not None:
            drain()                              # every outstanding result is on the host before the region ends
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        barrier()
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    for _ in range(max(args.warmup, 3)):
        step_resident()
    clocks.mark()
    n0 = ops.launch_count()
    total_ms = timed(step_resident, args.steps)
    launches = ops.launch_count() - n0
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:          # before the next step clears .grad
        dump_outputs(args.dump_outputs, train_step_outputs(torch, last["loss"], last["logits"], params))
    step_e2e()
    e2e_ms = timed(step_e2e, args.steps, meter.total)
    import math
    assert meter.count == args.steps + 1 and math.isfinite(meter.total())            # every step's loss was read
    step_e2e_sync()
    e2e_sync_ms = timed(step_e2e_sync, args.steps)

    # ---- roofline of the dominant kernel family (tcgen05 tap-GEMM), one extra profiled step -----------
    # The timed region above overlaps the weight-gradient GEMMs with the input-gradient chain on a second stream
    # (engine.WGRAD_STREAM): an event pair around a launch would then include the time it waits for SMs.  The profiled
    # step therefore runs every kernel on ONE stream, so that each launch's duration is its own.
    from importlib import import_module as _im
    _eng = _im("htr-vt_b200.engine")
    _ws, _eng.WGRAD_STREAM = _eng.WGRAD_STREAM, False
    step_resident()                       # (first single-stream step: fresh packed-weight tensors, untimed)
    ops.PROFILE = []
    step_resident()
    torch.cuda.synchronize()
    prof, ops.PROFILE = ops.PROFILE, None
    _eng.WGRAD_STREAM = _ws
    by = {}
    for name, fl, a, b in prof:
        d = by.setdefault(name, [0.0, 0.0, 0])
        d[0] += a.elapsed_time(b)
        d[1] += fl
        d[2] += 1
    gemm_names = ("gemm_tn", "gemm_nn", "linear_wgrad", "conv_fwd", "conv_dgrad", "conv_dgrad_bn", "conv_wgrad", "conv_wgrad_acc",
                  "conv_wgrad_acc_t", "conv_wgrad_acc_w")
    g_ms = sum(by[n][0] for n in gemm_names if n in by)
    g_fl = sum(by[n][1] for n in gemm_names if n in by)
    g_n = sum(by[n][2] for n in gemm_names if n in by)
    all_ms = sum(v[0] for v in by.values())

    # BASELINE config 4 at this N (every rank takes part: max-over-ranks timing between barriers)
    infer = None
    if not args.no_extras:
        try:
            infer = inference_metrics(torch, dist, dev, h, ops, model, world, rank, steps=5)
        except Exception as e:
            infer = {"error": repr(e)[:200]}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = load_peaks()
    # DRAM bytes of the tap-GEMM launches of one step: STATIC, from the committed ncu counters of this build's profile
    # run (profiles/*_traffic.json, `tools/ncu_step.sh`) - hardware counters cannot be read inside an unprofiled run
    traffic, traffic_src = None, None
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", name)))["tapgemm_dram_bytes_per_step"]
            traffic_src = "static from profiles/" + name
            break
        except Exception:
            pass
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback (B200_PROFILING.md sustained)"
    ach_tf = g_fl / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
    ms_step = total_ms / args.steps
    value = world * B / (ms_step * 1e-3)
    e2e_value = world * B / (e2e_ms / args.steps * 1e-3)
    h2d = img_h.numel() * 4 + tg_h.numel() * 4 + tl_h.numel() * 4
    line = {
        "metric": "line images/sec (train step)", "value": value, "unit": "img/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "v1_train_step_b128_64x512_c80", "batch_per_gpu": B, "img": [1, IMG_H, IMG_W],
                   "nb_cls": NB_CLS, "mask_ratio": MASK_RATIO, "max_span": MAX_SPAN,
                   "parallelism": "dp%d" % world,
                   "l2": "per-step working set (activations ~7 GB) >> 126 MB L2; no flush needed",
                   "algorithmic_tflop_per_step": 3 * GFLOP_FWD_PER_IMG * B / 1e3},
        "clocks": clk,
        "e2e": {"value": e2e_value, "unit": "img/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": e2e_ms / args.steps,
                "how": "pinned host batch -> HostPrefetcher (H2D of step i+1 under step i) -> model.forward -> CTCLoss -> "
                       "backward -> RunningLoss.add(loss): every step's loss is copied to pinned host memory and summed "
                       "on the host, the last ones inside the timed region; no per-step device sync",
                "sync_every_step": {"value": world * B / (e2e_sync_ms / args.steps * 1e-3),
                                    "ms_per_step": e2e_sync_ms / args.steps,
                                    "how": "the same with train.py:129's `loss.item()` every step"}},
        "gpu_launches": launches,
        "roofline": {"bound": "tensor", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": ach_tf / peak_tf if peak_tf else None, "traffic": traffic,
                     "traffic_note": "%s: ncu dram bytes (read + write) summed over the family's launches of one step; "
                                     "algorithmic = flops, the operands are re-read from L2" % traffic_src,
                     "kernel": "tapgemm_kernel (all conv / linear fwd, dgrad, wgrad launches of one step)",
                     "launches": g_n, "ms_in_step": g_ms, "share_of_step": g_ms / all_ms if all_ms else None,
                     "timing": "CUDA events around every launch of one extra step with all kernels on one stream "
                               "(sum over the family's launches; the timed steps overlap the weight-gradient GEMMs "
                               "on a second stream, where an event pair would include queueing); share_of_step is "
                               "relative to the sum of all launches of that single-stream step (%.3f ms)" % all_ms,
                     "peak_source": peak_src},
        "breakdown_ms": {k: round(v[0], 3) for k, v in sorted(by.items(), key=lambda kv: -kv[1][0])},
    }
    line["config"]["precision"] = ("16-bit tensor-core operands, fp32 accumulation: bf16 everywhere except the forward "
                                   "stem tensors (activations, raw conv outputs, forward conv weights), which are fp16 "
                                   "- same width and MMA rate, 3 more mantissa bits (train-mode parity, DESIGN.md 4)")
    if infer is not None:
        line["inference"] = infer
    if world == 1 and not args.no_extras:
        line["extra"] = extra_metrics(torch, dev, h, ops, H, model, peaks)
        try:
            line["extra"]["gpu_eager_baseline"] = gpu_eager_baseline(torch, dev)
        except Exception as e:
            line["extra"]["gpu_eager_baseline"] = {"error": repr(e)[:200]}
    if world == 1 and not args.no_cpu_baseline:
        rate, per, threads = cpu_reference_rate(20, 1, B=8)          # ~10 s of host work
        line["cpu_baseline"] = {"value": rate, "unit": "img/s", "cores": threads, "kind": "port",
                                "sample": "oracle port of model_v1 fwd+bwd+CTCLoss on 8 images/step, 20 timed steps"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=128, help="images per GPU")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train", choices=["train", "infer"],
                    help="train: fwd+bwd+CTC step, batch 128/GPU (headline, BASELINE configs 2-3); "
                         "infer: eval forward + greedy decode, 512 lines/GPU (config 4)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the CTC / inference / window-variant side metrics")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (train: loss, logits, gradient norms "
                         "and a seeded gradient sample; infer: logits, ids, lengths) as DIR/<name>.npy, rank 0 only; "
                         "bench_outputs/ in the checkout is git-ignored")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of this project's GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "infer":
        run_infer(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
