"""CPU test of TransFuse_S_adapt's HOST logic (module wiring, NHWC plumbing, gates, registration order / init) against goldens of
the unmodified reference (oracle/make_golden_transfuse_model.py): the C-ABI Functions are replaced by torch expressions of what
each kernel computes, so everything except the kernels themselves is checked here without a GPU.  The kernels are checked by
tests/test_transfuse_model_gpu.py."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from mdvit_b200 import ops, transfuse as T
from oracle import golden_sample as GS
from oracle.make_golden_transfuse_model import case, structure_loss_ref
from tests.helpers import fingerprint

GOLD = os.path.join(os.path.dirname(__file__), "golden", "transfuse_model_golden.npz")


from oracle.transfuse_oracle import (EmuBn as _EmuBn, EmuChannelPool as _EmuChannelPool, EmuConv as _EmuConv,      # noqa: E402,F401
                                     EmuGateCat as _EmuGateCat, EmuPool as _EmuPool, EmuResize as _EmuResize, deit_forward_torch)


@pytest.fixture()
def emulated(monkeypatch):
    monkeypatch.setattr(ops, "ConvBnActFn", _EmuConv)
    monkeypatch.setattr(ops, "BnActFn", _EmuBn)
    monkeypatch.setattr(ops, "MaxPool3s2Fn", _EmuPool)
    monkeypatch.setattr(ops, "ResizeACFn", _EmuResize)
    monkeypatch.setattr(ops, "GateCatFn", _EmuGateCat)
    monkeypatch.setattr(ops, "ChannelPoolFn", _EmuChannelPool)
    monkeypatch.setattr(T.DeiT_adapt, "forward", lambda self, imgs, label: deit_forward_torch(self, imgs, label))


def test_constructor_reproduces_reference_keys_and_init():
    g = np.load(GOLD)
    torch.manual_seed(0)
    m = T.TransFuse_S_adapt(drop_rate=0.0)
    assert list(m.state_dict().keys()) == list(g["keys"])
    # bit-identical weights: the fingerprints are float64 sums whose last bits depend on the host CPU's summation order, so they
    # must agree to 1e-12 of each tensor's norm (a zero tensor's fingerprint is exactly zero)
    fp, ref = fingerprint(list(m.named_parameters())), g["init_fp"]
    assert (np.abs(fp - ref).max(axis=1) <= 1e-12 * ref[:, 0]).all()


def test_wiring_matches_reference_forward_backward_on_cpu(emulated):
    g = np.load(GOLD)
    torch.manual_seed(0)
    m = T.TransFuse_S_adapt(drop_rate=0.0).train()
    img, mask, dlab = case()
    maps = m(img, dlab)
    for n, p in zip(("map_x", "map_1", "map_2"), maps):
        assert tuple(p.shape) == GS.shape(g, n)
        assert GS.rel_max(p, g, n) <= 2e-4, n
    losses = [structure_loss_ref(p, mask) for p in maps]
    loss = 0.5 * losses[2] + 0.3 * losses[1] + 0.2 * losses[0]
    np.testing.assert_allclose([l.item() for l in losses] + [loss.item()], g["losses"], rtol=2e-5)
    loss.backward()
    named = [(n, p.grad) for n, p in m.named_parameters() if p.grad is not None]
    assert [n for n, _ in named] == list(g["grad_names"])      # the same parameters are reached (skip_layer of square Residuals is not)
    fp, ref_fp = fingerprint(named), g["grad_fp"]
    # (conv biases in front of a BatchNorm have an exactly-zero true gradient: round-off there is compared on an absolute scale)
    err = np.abs(fp - ref_fp).max(axis=1) / (ref_fp[:, 0] + 1e-3 * np.median(ref_fp[:, 0]))
    # (the single-channel conv + BatchNorm2d(1) pairs in front of a sigmoid have cancellation-residue gradients: looser bound)
    ill = np.asarray([(".psi." in n) or (".spatial." in n) for n, _ in named])
    assert err[~ill].max() < 2e-2, (named[int(np.argmax(np.where(ill, 0, err)))][0], err[~ill].max())
    assert err[ill].max() < 0.2
    for k in g.files:
        if k.startswith("buf."):
            np.testing.assert_allclose(m.state_dict()[k[4:]].numpy(), g[k], rtol=1e-4, atol=1e-6)
    assert all(int(v) == 1 for k, v in m.state_dict().items() if k.endswith("num_batches_tracked") and "skip_layer" not in k
               and "layer4" not in k), "every BatchNorm that ran counts one batch"


def test_stacked_multi_dataset_forward_equals_consecutive_forwards(emulated):
    """TransFuse_S_adapt.forward_multi (all dataset mini-batches in one pass, BatchNorm per group) == one forward per dataset
    (multi_train_TransFuse.py:151-172), including every BatchNorm running statistic — host logic of the grouped path."""
    img, _, dlab = case(B=4, side=64)
    outs, bufs = [], []
    for stacked in (True, False):
        torch.manual_seed(0)
        m = T.TransFuse_S_adapt(drop_rate=0.0).train()
        with torch.no_grad():
            m.transformer.pos_embed = torch.nn.Parameter(0.02 * torch.randn(1, 16, 384))      # 64 x 64 images: 4 x 4 tokens
            if stacked:
                maps = m.forward_multi(img, dlab, 2)
            else:
                parts = [m(img[:2], dlab[:2]), m(img[2:], dlab[2:])]
                maps = [torch.cat([a, b]) for a, b in zip(*parts)]
        outs.append(maps)
        bufs.append({k: v.clone() for k, v in m.state_dict().items() if "running" in k or "num_batches" in k})
    for a, b in zip(*outs):
        assert torch.allclose(a, b, rtol=1e-4, atol=1e-5)
    for k in bufs[0]:
        assert torch.allclose(bufs[0][k].float(), bufs[1][k].float(), rtol=1e-4, atol=1e-6), k


def test_trainer_stacked_loss_equals_per_dataset_losses(emulated, monkeypatch):
    """TransFuseTrainer host logic: the stacked schedule back-propagates G x mean(per-sample terms over the whole stack) and reports
    group means — the same numbers as one forward + three structure losses per dataset (multi_train_TransFuse.py:151-172,191),
    and the same gradients."""
    from mdvit_b200.train_step import TransFuseTrainer
    from oracle.make_golden_transfuse_model import structure_loss_ref

    def weit_ref(mask):
        return 1 + 5 * torch.abs(F.avg_pool2d(mask, kernel_size=31, stride=1, padding=15) - mask)

    def loss_ref(pred, mask, weit=None, per_sample=False):
        weit = weit_ref(mask) if weit is None else weit
        wbce = (weit * F.binary_cross_entropy_with_logits(pred, mask, reduction="none")).sum(dim=(2, 3)) / weit.sum(dim=(2, 3))
        p = torch.sigmoid(pred)
        inter, union = ((p * mask) * weit).sum(dim=(2, 3)), ((p + mask) * weit).sum(dim=(2, 3))
        ps = (wbce + 1 - (inter + 1) / (union - inter + 1)).flatten()
        return (ps.mean(), ps.detach()) if per_sample else ps.mean()

    monkeypatch.setattr(ops, "structure_weit", weit_ref)
    monkeypatch.setattr(ops, "structure_loss", loss_ref)
    img, mask, _ = case(B=4, side=64)
    assert abs(loss_ref(img[:, :1], mask).item() - structure_loss_ref(img[:, :1], mask).item()) < 1e-6
    batches = [(img[:2], mask[:2], 1), (img[2:], mask[2:], 3)]
    res = []
    for fused in (True, False):
        torch.manual_seed(0)
        m = T.TransFuse_S_adapt(drop_rate=0.0).train()
        with torch.no_grad():
            m.transformer.pos_embed = torch.nn.Parameter(0.02 * torch.randn(1, 16, 384))      # 64 x 64 images: 4 x 4 tokens
        tr = TransFuseTrainer(m, fuse_datasets=fused)
        losses = tr.forward_losses(batches)
        total = tr._total_loss if tr._total_loss is not None else losses.sum()
        assert (tr._total_loss is not None) == fused
        total.backward()
        assert len(tr.last_logits) == 2 and tuple(tr.last_logits[0].shape) == (2, 1, 64, 64)
        res.append((losses.detach().clone(), total.item(), tr.grad.clone()))
    (l0, t0, g0), (l1, t1, g1) = res
    assert torch.allclose(l0, l1, rtol=1e-4) and abs(t0 - t1) < 1e-4 * abs(t1) and abs(t0 - l0.sum().item()) < 1e-4 * abs(t0)
    assert ((g0 - g1).norm() / g1.norm()).item() < 2e-2      # (fp32 reordering through this ill-conditioned net, see DESIGN.md section 11)
