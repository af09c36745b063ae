"""Development aid: TransFuse_S_adapt forward + backward + structure_loss at B images of 256 x 256 on one GPU — this repo's kernels
vs the same module evaluated by stock PyTorch (cuDNN convolutions, aten BatchNorm / pooling / resize, SDPA-free DeiT) on the same
weights, and the parity margins against the reference goldens.  python scripts/dev_transfuse_time.py [B]"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mdvit_b200 import _lib as L, ops, transfuse as T      # noqa: E402
from oracle import golden_sample as GS      # noqa: E402
from oracle.make_golden_transfuse_model import case      # noqa: E402
from tests import test_transfuse_wiring as W      # noqa: E402
from tests.helpers import fingerprint      # noqa: E402


def step(m, img, mask, dlab, mine):
    maps = m(img, dlab)
    if mine:
        weit = ops.structure_weit(mask)
        losses = [ops.structure_loss(p, mask, weit) for p in maps]
    else:
        from oracle.make_golden_transfuse_model import structure_loss_ref
        losses = [structure_loss_ref(p, mask) for p in maps]
    loss = 0.5 * losses[2] + 0.3 * losses[1] + 0.2 * losses[0]
    loss.backward()
    return maps, losses, loss


def timed(fn, n=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(n):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / n


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
    dev = torch.device("cuda")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    g = np.load(os.path.join(ROOT, "tests", "golden", "transfuse_model_golden.npz"))
    torch.manual_seed(0)
    m = T.TransFuse_S_adapt(drop_rate=0.0).to(dev).train()
    img, mask, dlab = (t.to(dev) for t in case())
    maps, losses, loss = step(m, img, mask, dlab, True)
    torch.cuda.synchronize()
    for n, p in zip(("map_x", "map_1", "map_2"), maps):
        print(f"{n}: rel err {GS.rel_max(p, g, n):.3e}")
    print("losses", [round(l.item(), 6) for l in losses], loss.item(), "golden", g["losses"])
    named = [(n, p.grad) for n, p in m.named_parameters() if p.grad is not None]
    fp, ref_fp = fingerprint(named), g["grad_fp"]
    floor = 1e-3 * np.median(ref_fp[:, 0])
    err = np.abs(fp[:, 0] - ref_fp[:, 0]) / (ref_fp[:, 0] + floor)
    order = np.argsort(-err)
    print("grad-norm rel err: max %.3e median %.3e; worst:" % (err.max(), np.median(err)), [(named[i][0], round(float(err[i]), 4)) for i in order[:8]])
    for k in g.files:
        if k.startswith("grad."):
            got, ref = dict(named)[k[5:]], torch.from_numpy(g[k]).to(dev)
            print(f"  {k}: {((got - ref).abs().max() / (ref.abs().max() + 1e-30)).item():.3e} (absmax {ref.abs().max().item():.2e})")
    # ---- timing at batch B
    img = torch.randn(B, 3, 256, 256, device=dev)
    mask = (torch.rand(B, 1, 256, 256, device=dev) > 0.5).float()
    dlab = torch.nn.functional.one_hot(torch.arange(B, device=dev) % 4, 4).float()

    def run_mine():
        m.zero_grad(set_to_none=True)
        step(m, img, mask, dlab, True)

    n0 = L.lib().mdv_launch_count()
    run_mine()
    print("library launches per forward+backward:", L.lib().mdv_launch_count() - n0)
    t_mine = timed(run_mine)
    print(f"mdvit_b200: {t_mine:.2f} ms per forward+backward at B={B} -> {B / t_mine * 1e3:.0f} images/s")
    if os.environ.get("MDV_PROFILE"):
        L.PROFILE_LOG.clear()
        run_mine()
        print(L.profile_report(40))
    # ---- the same module through stock PyTorch
    for name, cls in (("ConvBnActFn", W._EmuConv), ("BnActFn", W._EmuBn), ("MaxPool3s2Fn", W._EmuPool), ("ResizeACFn", W._EmuResize),
                     ("GateCatFn", W._EmuGateCat), ("ChannelPoolFn", W._EmuChannelPool)):
        setattr(ops, name, cls)
    T.DeiT_adapt.forward = lambda self, imgs, label: W.deit_forward_torch(self, imgs, label)

    def run_torch():
        m.zero_grad(set_to_none=True)
        step(m, img, mask, dlab, False)

    t0 = time.time()
    t_fp32 = timed(run_torch, n=3, warm=1)
    print(f"stock PyTorch eager fp32: {t_fp32:.2f} ms -> {B / t_fp32 * 1e3:.0f} images/s  ({time.time() - t0:.1f} s wall)")
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    t_tf32 = timed(run_torch, n=3, warm=1)
    print(f"stock PyTorch eager TF32: {t_tf32:.2f} ms -> {B / t_tf32 * 1e3:.0f} images/s")

    def run_amp():
        m.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            maps = m(img, dlab)
        from oracle.make_golden_transfuse_model import structure_loss_ref
        ls = [structure_loss_ref(p.float(), mask) for p in maps]
        (0.5 * ls[2] + 0.3 * ls[1] + 0.2 * ls[0]).backward()

    t_amp = timed(run_amp, n=3, warm=1)
    print(f"stock PyTorch eager bf16 autocast: {t_amp:.2f} ms -> {B / t_amp * 1e3:.0f} images/s")


if __name__ == "__main__":
    main()
