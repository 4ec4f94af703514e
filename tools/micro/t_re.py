import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch.nn.functional as F
from importlib import import_module
import htrvt_b200
o = import_module("htr-vt_b200.ops")
torch.manual_seed(4)
torch.backends.cudnn.allow_tf32 = False
NB, H, W, Cin, Cout, ks, sh, sw = 2, 8, 512, 192, 192, 3, 1, 1
x = torch.randn(NB, H, W, Cin, device="cuda").bfloat16()
w = (torch.randn(Cout, Cin, ks, ks, device="cuda") / (Cin * 9) ** 0.5).bfloat16()
wk = w.permute(0, 2, 3, 1).reshape(Cout, 9, Cin).contiguous()
yr = F.conv2d(x.float().permute(0, 3, 1, 2), w.float(), None, (sh, sw), 1)
y = o.conv_fwd(x, wk, ks, sh, sw)
d = (y.permute(0, 3, 1, 2).float() - yr).abs()
print("max err", float(d.max()), "ref max", float(yr.abs().max()))
# which taps are wrong? use a weight with a single tap active
for t in range(9):
    w1 = torch.zeros_like(w); w1[:, :, t // 3, t % 3] = w[:, :, t // 3, t % 3]
    wk1 = w1.permute(0, 2, 3, 1).reshape(Cout, 9, Cin).contiguous()
    yr1 = F.conv2d(x.float().permute(0, 3, 1, 2), w1.float(), None, (sh, sw), 1)
    y1 = o.conv_fwd(x, wk1, ks, sh, sw)
    d1 = (y1.permute(0, 3, 1, 2).float() - yr1).abs()
    # per output column error profile
    col = d1.amax(dim=(0, 1, 2))
    print("tap", t, "max err %.3f" % float(d1.max()), "cols with err:", int((col > 0.05).sum()), "first bad cols", (col > 0.05).nonzero().flatten()[:6].tolist())
