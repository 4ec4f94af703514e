"""Timing of fc2's input-gradient GEMM with the fused activation backward (EPI 4) against the plain GEMM."""
import sys, os, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from importlib import import_module
import htrvt_b200
o = import_module("htr-vt_b200.ops")
torch.manual_seed(0)
M, Kd, N = 16384, 768, 3072
dy = torch.randn(M, Kd, device="cuda").bfloat16()
w2 = (torch.randn(Kd, N, device="cuda") / Kd ** 0.5).bfloat16()
gd = torch.rand(M, N, device="cuda").bfloat16()
du = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
bg = torch.zeros(N, device="cuda")
for _ in range(3): o.gemm_nn(dy, w2, du, gelu_u=gd, colsum=bg)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(20): o.gemm_nn(dy, w2, du, gelu_u=gd, colsum=bg)
e1.record(); torch.cuda.synchronize()
print("fc2 dgrad * gelu' + colsum: %.1f us" % (e0.elapsed_time(e1) / 20 * 1e3))
ref = (dy.float() @ w2.float()) * gd.float()
print("rel err", float((du.float() - ref).abs().max() / ref.abs().max()))
da = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
e0.record()
for _ in range(20): o.gemm_nn(dy, w2, da)
e1.record(); torch.cuda.synchronize()
print("plain fc2 dgrad: %.1f us" % (e0.elapsed_time(e1) / 20 * 1e3))

