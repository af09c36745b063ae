"""Development aid (CPU, no GPU needed): how far does operand rounding alone move TransFuse_S_adapt from the fp32 reference goldens?
The module is evaluated in fp32 torch (the C-ABI Functions replaced by the torch expressions of tests/test_transfuse_wiring.py)
with the conv operands rounded to TF32 (10 mantissa bits) in the forward and / or the conv output gradients rounded to bf16
(7 bits) in the backward — nothing else differs from the run that produced the goldens.

    python scripts/dev_transfuse_rounding_sensitivity.py tf32|bf16bwd|both [traj]

DESIGN.md section 11 quotes: `tf32` moves the maps by 0.98e-2 / 0.9e-3 / 1.7e-2 of abs-max and resnet.conv1.weight's gradient by 24 %
max-abs; `both traj` ends the 5-step trajectory 3-4 % (loss) / 1.6e-2 (Dice) from the reference."""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mdvit_b200 import ops, transfuse as T      # noqa: E402
from oracle import golden_sample as GS      # noqa: E402
from oracle.make_golden_randinit import hard_dice      # noqa: E402
from oracle.make_golden_transfuse_model import case, structure_loss_ref      # noqa: E402
from tests import test_transfuse_wiring as W      # noqa: E402

mode = sys.argv[1] if len(sys.argv) > 1 else "both"


def rnd(t, bits):
    """round to `bits` explicit mantissa bits (10 = TF32, 7 = bf16)"""
    sh = 23 - bits
    i = t.contiguous().view(torch.int32)
    return (((i + (1 << (sh - 1))) >> sh) << sh).view(torch.float32)


class RoundFwd(torch.autograd.Function):
    @staticmethod
    def forward(ctx, t, bits):
        return rnd(t, bits)

    @staticmethod
    def backward(ctx, g):
        return g, None


class RoundBwd(torch.autograd.Function):
    @staticmethod
    def forward(ctx, t, bits):
        ctx.bits = bits
        return t.view_as(t)

    @staticmethod
    def backward(ctx, g):
        return rnd(g, ctx.bits), None


class RoundedConv:
    @staticmethod
    def apply(x, w, cbias, *a):
        if mode in ("tf32", "both"):
            x, w = RoundFwd.apply(x, 10), RoundFwd.apply(w, 10)
        y = W._EmuConv.apply(x, w, cbias, *a)
        return RoundBwd.apply(y, 7) if mode in ("bf16bwd", "both") else y


for name, cls in (("ConvBnActFn", RoundedConv), ("BnActFn", W._EmuBn), ("MaxPool3s2Fn", W._EmuPool), ("ResizeACFn", W._EmuResize),
                  ("GateCatFn", W._EmuGateCat), ("ChannelPoolFn", W._EmuChannelPool)):
    setattr(ops, name, cls)
T.DeiT_adapt.forward = lambda self, imgs, label: W.deit_forward_torch(self, imgs, label)
torch.manual_seed(0)
m = T.TransFuse_S_adapt(drop_rate=0.0).train()

if len(sys.argv) > 2 and sys.argv[2] == "traj":
    from oracle.make_golden_transfuse_traj import LR, STEPS, WD, batches
    g = np.load(os.path.join(ROOT, "tests", "golden", "transfuse_traj_golden.npz"))
    opt = torch.optim.AdamW(m.parameters(), lr=LR, weight_decay=WD)
    for step in range(STEPS):
        ls, ds = [], []
        for img, mask, d in batches():
            dl = F.one_hot(torch.full((img.shape[0],), d), 4).float()
            mx, m1, m2 = m(img, dl)
            ls.append(0.5 * structure_loss_ref(m2, mask) + 0.3 * structure_loss_ref(m1, mask) + 0.2 * structure_loss_ref(mx, mask))
            ds.append(hard_dice(m2.detach(), mask))
        opt.zero_grad()
        sum(ls).backward()
        opt.step()
        print(step, "loss", [round(l.item(), 4) for l in ls], "ref", g["losses"][step].round(4), "dice", [round(x, 4) for x in ds], "ref", g["dice"][step].round(4))
    sys.exit(0)

g = np.load(os.path.join(ROOT, "tests", "golden", "transfuse_model_golden.npz"))
img, mask, dlab = case()
maps = m(img, dlab)
for n, p in zip(("map_x", "map_1", "map_2"), maps):
    print(n, "max-abs / abs-max", GS.rel_max(p, g, n))
ls = [structure_loss_ref(p, mask) for p in maps]
(0.5 * ls[2] + 0.3 * ls[1] + 0.2 * ls[0]).backward()
named = dict((n, p.grad) for n, p in m.named_parameters() if p.grad is not None)
for k in g.files:
    if k.startswith("grad."):
        got = named[k[5:]]
        print(f"  {k}: max-abs {GS.rel_max(got, g, k):.3e}  rel-L2 {GS.rel_l2(got, g, k):.3e}")
