import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import numpy as np, torch
from functools import partial
from importlib import import_module
import htrvt_b200 as h
H = import_module("htr-vt_b200.model.HTR_VT")
dev = torch.device("cuda", 0)
nb_cls, W, D, depth, heads, Bs = 24, 128, 256, 2, 2, 4
torch.manual_seed(100)
m = H.MaskedAutoencoderViT(nb_cls, img_size=[64, W], patch_size=(4, 64), embed_dim=D, depth=depth, num_heads=heads, mlp_ratio=4, norm_layer=partial(torch.nn.LayerNorm, eps=1e-6)).to(dev).train()
rs = np.random.RandomState(0)
imgs = torch.from_numpy(rs.rand(2 * Bs, 1, 64, W).astype(np.float32))
lens = rs.randint(3, 9, size=2 * Bs).astype(np.int32)
tgs = rs.randint(1, nb_cls, size=int(lens.sum())).astype(np.int32)
offs = np.concatenate([[0], np.cumsum(lens)])
def step(r):
    for p in m.parameters(): p.grad = None
    lo, hi = r * Bs, (r + 1) * Bs
    x, tg, tl = imgs[lo:hi].to(dev), torch.from_numpy(tgs[offs[lo]:offs[hi]]).to(dev), torch.from_numpy(lens[lo:hi])
    torch.manual_seed(5)
    preds = m(x, 0.4, 8, use_masking=True)
    h.ctc_loss_from_logits(preds.float(), tg, tl).mean().backward()
    return preds.detach().clone(), {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}
pa, ga = step(0); pb, gb = step(0)
print('forward equal', torch.equal(pa, pb))
rows = sorted(((float((ga[n]-gb[n]).abs().max()/(ga[n].abs().max()+1e-20)), n) for n in ga), reverse=True)
for e, n in rows[:10]: print('%.3e %s' % (e, n))
