"""TransFuse_S_adapt (BASELINE.json config 4 / SURVEY 8 f-1) on the GPU, through the C ABI:
 * op level — dense conv (+BN, +residual, +ReLU), max-pool, align_corners resize, structure_loss against plain torch fp32 of the
   same op (TF32 forward GEMMs: 2e-3 of the abs-max; bf16 gradient GEMMs: 2e-2);
 * model level — the three logit maps, the deep-supervision loss, every parameter-gradient norm and the BatchNorm running
   statistics against goldens of the UNMODIFIED reference at its own random init (oracle/make_golden_transfuse_model.py)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import golden_sample as GS
from oracle.make_golden_transfuse_model import case, structure_loss_ref
from tests.helpers import fingerprint
from tests.test_transfuse_wiring import _EmuConv

GOLD = os.path.join(os.path.dirname(__file__), "golden", "transfuse_model_golden.npz")
LOSS_GOLD = os.path.join(os.path.dirname(__file__), "golden", "transfuse_structure_loss_golden.npz")
pytestmark = pytest.mark.gpu
FWD_TOL, BWD_TOL = 2e-3, 2e-2


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return torch.device("cuda")


def rel(a, b):
    a, b = torch.as_tensor(a).float().cpu(), torch.as_tensor(b).float().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-30)).item()


def rel_l2(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def tf32_representable(t):
    """round to 10 explicit mantissa bits: products of such operands are exact on the TF32 tensor-core path AND in fp32, so the
    op-level comparison below sees the same pre-activations (no ReLU-mask flips on near-zero values) and isolates the kernels"""
    i = t.contiguous().view(torch.int32)
    return (((i + (1 << 12)) >> 13) << 13).view(torch.float32)


# (Cin, Cout, k, stride, H, W, bn, act, residual, nchw, bias)
CONV_CASES = [
    (64, 64, 3, 1, 16, 16, True, True, False, False, False),      # BasicBlock conv1
    (64, 64, 3, 1, 16, 16, True, True, True, False, False),       # BasicBlock conv2 + identity
    (64, 128, 3, 2, 16, 16, True, True, False, False, False),     # layer2.0.conv1 (stride 2)
    (64, 128, 1, 2, 16, 16, True, False, False, False, False),    # layer2.0.downsample
    (3, 64, 7, 2, 32, 32, True, True, False, True, False),        # resnet.conv1 on the NCHW image
    (2, 1, 7, 1, 16, 16, False, False, False, False, False),      # BiFusion_block.spatial.conv
    (64, 1, 3, 1, 16, 16, False, False, False, False, True),      # output heads
    (128, 1, 1, 1, 8, 8, False, False, False, False, True),       # Attention_block.psi
    (384, 128, 1, 1, 8, 8, True, False, False, False, True),      # W_x / identity convs
    (128, 128, 1, 1, 8, 8, True, True, True, False, True),        # relu(g1 + x1)
    (64, 128, 1, 1, 8, 12, False, False, True, False, True),      # Residual.conv3 + residual (GEMM epilogue add)
    (192, 64, 3, 1, 12, 8, True, True, False, False, True),       # DoubleConv first conv, ragged map (im2col fallback)
    (64, 64, 3, 1, 64, 64, True, True, False, False, False),      # implicit GEMM, 2 image rows per 128-row tile
    (128, 128, 3, 1, 32, 32, True, True, True, False, False),     # implicit GEMM, 4 rows per tile, + identity
    (256, 256, 3, 1, 16, 16, True, True, False, False, False),    # implicit GEMM, 8 rows per tile (2 tiles per image)
    (384, 128, 3, 1, 32, 32, True, True, False, False, True),     # up1 / up_c_1_2 DoubleConv
    (32, 32, 3, 1, 64, 64, True, True, False, False, True),       # Residual.conv2 of up_c_2_1: implicit forward, im2col input gradient
]


@pytest.mark.parametrize("pair", [-1, 1])
@pytest.mark.parametrize("case_", CONV_CASES)
def test_conv_bn_act_fwd_bwd_vs_torch(case_, pair):
    from mdvit_b200 import _lib as L, ops
    dev = _dev()
    if pair == 1 and case_[2] != 3:
        pytest.skip("the forced CTA-pair run covers the 3x3 convolutions")
    L.lib().mdv_gemm_force_pair(pair)      # 1: every NT GEMM (implicit-conv mode included) as tcgen05 cta_group::2 CTA pairs
    try:
        _conv_case(case_, dev, ops)
    finally:
        L.lib().mdv_gemm_force_pair(-1)


def _conv_case(case_, dev, ops):
    Cin, Cout, k, s, H, W, bn, act, res, nchw, bias = case_
    B = 3
    g = torch.Generator().manual_seed(k * 1000 + Cin + Cout)
    x = tf32_representable(torch.randn((B, Cin, H, W) if nchw else (B, H * W, Cin), generator=g)).to(dev).requires_grad_(not nchw)
    w = tf32_representable(torch.randn((Cout, Cin, k, k), generator=g) / (Cin * k * k) ** 0.5).to(dev).requires_grad_(True)
    cb = (0.3 * torch.randn(Cout, generator=g)).to(dev).requires_grad_(True) if bias else None
    gam = (1 + 0.2 * torch.randn(Cout, generator=g)).to(dev).requires_grad_(True) if bn else None
    bet = (0.2 * torch.randn(Cout, generator=g)).to(dev).requires_grad_(True) if bn else None
    Ho, Wo, _ = ops.conv_geom(H, W, k, s)
    r = torch.randn((B, Ho * Wo, Cout), generator=g).to(dev).requires_grad_(True) if res else None
    probe = torch.randn((B, Ho * Wo, Cout), generator=g).to(dev)
    a = ops.ACT_RELU if act else ops.ACT_NONE
    outs = []
    for fn in (ops.ConvBnActFn, _EmuConv):
        bufs = (torch.zeros(Cout, device=dev), torch.ones(Cout, device=dev), torch.zeros((), dtype=torch.long, device=dev)) if bn else None
        for t in (x, w, cb, gam, bet, r):
            if t is not None:
                t.grad = None
        y = fn.apply(x, w, cb, gam, bet, r, bufs, B, H, W, s, a, True, nchw)
        (y * probe).sum().backward()
        outs.append((y.detach(), [None if (t is None or t.grad is None) else t.grad.clone() for t in (x, w, cb, gam, bet, r)], bufs))
    (y0, g0, b0), (y1, g1, b1) = outs
    assert rel(y0, y1) < FWD_TOL
    for name, a_, b_ in zip(("dx", "dw", "dbias", "dgamma", "dbeta", "dres"), g0, g1):
        assert (a_ is None) == (b_ is None), name
        if a_ is None:
            continue
        if name == "dbias" and bn:      # exactly zero in exact arithmetic (BatchNorm removes the bias): only round-off to compare
            assert torch.isfinite(a_).all()
            continue
        # L2-relative: with K up to 3456 the two fp32 accumulation orders can still put a BatchNorm output on different sides of
        # zero (about one ReLU-mask flip per few 1e5 elements), which moves a handful of gradient entries by a whole weight
        assert rel_l2(a_, b_) < BWD_TOL, (name, rel_l2(a_, b_))
        big = ((a_ - b_).abs() > 5 * BWD_TOL * b_.abs().max()).float().mean().item()
        assert big < 2e-3, (name, big)
    if bn:
        assert rel(b0[0], b1[0]) < FWD_TOL and rel(b0[1], b1[1]) < FWD_TOL and int(b0[2]) == 1


def test_bn_act_fn_vs_torch():
    from mdvit_b200 import ops
    dev = _dev()
    B, N, C = 3, 96, 192
    x = torch.randn(B, N, C, device=dev).requires_grad_(True)
    gam, bet = (1 + 0.2 * torch.randn(C, device=dev)).requires_grad_(True), (0.2 * torch.randn(C, device=dev)).requires_grad_(True)
    probe = torch.randn(B, N, C, device=dev)
    res = []
    for mine in (True, False):
        bufs = (torch.zeros(C, device=dev), torch.ones(C, device=dev), torch.zeros((), dtype=torch.long, device=dev))
        for t in (x, gam, bet):
            t.grad = None
        if mine:
            y = ops.BnActFn.apply(x, gam, bet, bufs, ops.ACT_RELU, True)
        else:
            y = torch.relu(F.batch_norm(x.transpose(1, 2), bufs[0], bufs[1], gam, bet, True, 0.1, 1e-5).transpose(1, 2))
        (y * probe).sum().backward()
        res.append((y.detach(), x.grad.clone(), gam.grad.clone(), bet.grad.clone()))
    for a_, b_ in zip(*res):
        assert rel(a_, b_) < 1e-4


@pytest.mark.parametrize("shape", [(2, 16, 16, 64), (3, 10, 14, 8), (1, 7, 9, 4)])
def test_maxpool_fwd_bwd_exact(shape):
    from mdvit_b200 import ops
    dev = _dev()
    B, H, W, C = shape
    x = torch.randn(B, H * W, C, device=dev)
    x = torch.relu(x)      # ties at zero, as after resnet's ReLU
    x.requires_grad_(True)
    y = ops.MaxPool3s2Fn.apply(x, H, W)
    xr = x.detach().view(B, H, W, C).permute(0, 3, 1, 2).clone().requires_grad_(True)
    yr = F.max_pool2d(xr, 3, 2, 1)
    assert torch.equal(y.view(B, yr.shape[2], yr.shape[3], C).permute(0, 3, 1, 2), yr)
    probe = torch.randn_like(yr)
    (yr * probe).sum().backward()
    (y * probe.permute(0, 2, 3, 1).reshape(B, -1, C)).sum().backward()
    gr = xr.grad.permute(0, 2, 3, 1).reshape(B, H * W, C)
    # ties (equal maxima inside a window) may be routed to a different tap than cuDNN's; away from ties the routing is identical
    tie = (x.detach() == 0)
    assert torch.allclose(x.grad[~tie], gr[~tie], rtol=1e-6, atol=1e-6)
    assert torch.allclose(x.grad.sum(), gr.sum(), rtol=1e-4)


@pytest.mark.parametrize("shape", [(2, 16, 16, 32, 32, 384), (2, 8, 8, 16, 16, 128), (3, 16, 16, 256, 256, 1), (2, 64, 64, 256, 256, 1),
                                   (1, 5, 7, 10, 14, 4)])
def test_resize_align_corners_fwd_bwd(shape):
    from mdvit_b200 import ops
    dev = _dev()
    B, H, W, Ho, Wo, C = shape
    x = torch.randn(B, H * W, C, device=dev).requires_grad_(True)
    y = ops.ResizeACFn.apply(x, H, W, Ho, Wo)
    xr = x.detach().view(B, H, W, C).permute(0, 3, 1, 2).clone().requires_grad_(True)
    yr = F.interpolate(xr, size=(Ho, Wo), mode="bilinear", align_corners=True)
    assert rel(y.view(B, Ho, Wo, C).permute(0, 3, 1, 2), yr) < 1e-5
    probe = torch.randn_like(yr)
    (yr * probe).sum().backward()
    (y * probe.permute(0, 2, 3, 1).reshape(B, -1, C)).sum().backward()
    assert rel(x.grad, xr.grad.permute(0, 2, 3, 1).reshape(B, H * W, C)) < 1e-5


def test_structure_loss_vs_reference_formula_and_golden():
    from mdvit_b200 import ops
    dev = _dev()
    g = np.load(LOSS_GOLD)          # the reference's three maps (fp16) with the loss and its gradient on them
    _, mask, _ = case()
    mask = mask.to(dev)
    weit = ops.structure_weit(mask)
    ref_weit = 1 + 5 * torch.abs(F.avg_pool2d(mask, kernel_size=31, stride=1, padding=15) - mask)
    assert rel(weit, ref_weit) < 1e-5
    for i, n in enumerate(("x", "1", "2")):
        pred = torch.from_numpy(g["pred_" + n].astype(np.float32)).to(dev).requires_grad_(True)
        loss = ops.structure_loss(pred, mask, weit)
        assert abs(loss.item() - g["losses"][i]) < 2e-5 * abs(g["losses"][i])
        coef = (0.2, 0.3, 0.5)[i]
        (coef * loss).backward()
        assert GS.rel_max(pred.grad, g, "dpred_" + n) < 1e-4
    # a saturated / random case against the formula itself
    pred = (8 * torch.randn(3, 1, 64, 64, device=dev)).requires_grad_(True)
    m2 = (torch.rand(3, 1, 64, 64, device=dev) > 0.6).float()
    l1 = ops.structure_loss(pred, m2)
    l1.backward()
    g1 = pred.grad.clone()
    pred.grad = None
    l2 = structure_loss_ref(pred, m2)
    l2.backward()
    assert abs(l1.item() - l2.item()) < 1e-5 * abs(l2.item()) and rel(g1, pred.grad) < 1e-4


def _run_model(m, batch, mine):
    from mdvit_b200 import ops
    img, mask, dlab = batch
    m.zero_grad(set_to_none=True)
    maps = m(img, dlab)
    if mine:
        weit = ops.structure_weit(mask)
        losses = [ops.structure_loss(p, mask, weit) for p in maps]
    else:
        losses = [structure_loss_ref(p, mask) for p in maps]
    loss = 0.5 * losses[2] + 0.3 * losses[1] + 0.2 * losses[0]      # multi_train_TransFuse.py:169-172
    loss.backward()
    torch.cuda.synchronize()
    grads = {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}
    return [p.detach().clone() for p in maps], [l.item() for l in losses] + [loss.item()], grads


@pytest.fixture(scope="module")
def trained_once():
    """One training forward + backward of TransFuse_S_adapt at the reference's random init on the golden batch: with this repo's
    kernels, and — the yardstick — the SAME module evaluated by stock PyTorch on the same GPU with its default numerics (cuDNN TF32
    convolutions).  The network at its random init is ill-conditioned (single-channel BatchNorms in front of sigmoids, 16 ReLU
    layers): rounding the conv operands to TF32 alone moves resnet.conv1's gradient by 22-25 % (measured on the CPU, DESIGN.md
    section 7), so the gradient bounds below are stated relative to what PyTorch's own GPU run of the reference would give."""
    import copy
    from mdvit_b200 import ops, transfuse as T
    from tests import test_transfuse_wiring as W
    dev = _dev()
    torch.manual_seed(0)
    m = T.TransFuse_S_adapt(drop_rate=0.0).to(dev).train()
    init = copy.deepcopy(m.state_dict())
    batch = tuple(t.to(dev) for t in case())
    mine = _run_model(m, batch, True)
    sd_after = copy.deepcopy(m.state_dict())
    with torch.no_grad():
        m.eval()
        emaps = [p.clone() for p in m(batch[0], batch[2])]
        m.train()
    # stock PyTorch, TF32 convolutions / matmuls allowed (its default for cuDNN), same initial state
    m.load_state_dict(init)
    saved = {n: getattr(ops, n) for n in ("ConvBnActFn", "BnActFn", "MaxPool3s2Fn", "ResizeACFn", "GateCatFn", "ChannelPoolFn")}
    fwd = T.DeiT_adapt.forward
    try:
        for n, c in (("ConvBnActFn", W._EmuConv), ("BnActFn", W._EmuBn), ("MaxPool3s2Fn", W._EmuPool), ("ResizeACFn", W._EmuResize),
                     ("GateCatFn", W._EmuGateCat), ("ChannelPoolFn", W._EmuChannelPool)):
            setattr(ops, n, c)
        T.DeiT_adapt.forward = lambda self, imgs, label: W.deit_forward_torch(self, imgs, label)
        torch.backends.cuda.matmul.allow_tf32 = True
        torch.backends.cudnn.allow_tf32 = True
        stock = _run_model(m, batch, False)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        T.DeiT_adapt.forward = fwd
        for n, c in saved.items():
            setattr(ops, n, c)
    return mine, stock, sd_after, emaps


def test_model_maps_and_losses_match_reference_golden(trained_once):
    g = np.load(GOLD)
    (maps, losses, _), (smaps, _, _), sd_after, _ = trained_once
    for n, p, sp in zip(("map_x", "map_1", "map_2"), maps, smaps):
        assert tuple(p.shape) == GS.shape(g, n)
        e, es = GS.rel_max(p, g, n), GS.rel_max(sp, g, n)
        print(f"{n}: ours {e:.3e}, stock PyTorch TF32 {es:.3e}")
        assert e < max(1e-2, 2.0 * es) and e < 3e-2, (n, e, es)
    np.testing.assert_allclose(losses, g["losses"], rtol=2e-3)
    for k in g.files:
        if k.startswith("buf."):
            assert rel(sd_after[k[4:]], g[k]) < 1e-2, k


def test_model_gradients_match_reference_golden(trained_once):
    g = np.load(GOLD)
    (_, _, grads), (_, _, sgrads), _, _ = trained_once
    assert list(grads.keys()) == list(g["grad_names"])
    assert all(torch.isfinite(t).all().item() for t in grads.values())
    ref_fp = g["grad_fp"]
    med = np.median(ref_fp[:, 0])

    def norm_err(gr):
        fp = fingerprint(list(gr.items()))
        # |norm - ref| relative to ref + 5 % of the median gradient norm: conv biases in front of a BatchNorm have an exactly-zero
        # true gradient (pure round-off), which this floor compares on an absolute scale
        return np.abs(fp[:, 0] - ref_fp[:, 0]) / (ref_fp[:, 0] + 5e-2 * med)

    err, serr = norm_err(grads), norm_err(sgrads)
    names = list(grads.keys())
    # the single-channel conv + BatchNorm2d(1) pairs (Attention_block.psi, BiFusion_block.spatial) sit in front of a sigmoid and
    # their gradients are cancellation residues: TF32 rounding alone moves them by up to > 100 % (also in stock PyTorch)
    ill = np.asarray([(".psi." in n) or (".spatial." in n) for n in names])
    print("grad-norm error: ours median %.3e p95 %.3e max(well-conditioned) %.3e; stock PyTorch TF32 median %.3e p95 %.3e max %.3e"
          % (np.median(err), np.percentile(err, 95), err[~ill].max(), np.median(serr), np.percentile(serr, 95), serr[~ill].max()))
    assert np.median(err) < 2e-2
    assert np.percentile(err, 95) < 0.1
    assert err[~ill].max() < max(0.1, 2.0 * serr[~ill].max()), (names[int(np.argmax(np.where(ill, 0, err)))], err[~ill].max())
    for k in g.files:
        if k.startswith("grad."):
            n = k[5:]
            if GS.absmax(g, k) < 1e-3 * med or ".psi.1." in n or ".spatial.bn." in n:
                continue
            e, es = GS.rel_max(grads[n], g, k), GS.rel_max(sgrads[n], g, k)
            print(f"{k}: ours {e:.3e}, stock PyTorch TF32 {es:.3e}")
            assert e < max(5e-2, 2.5 * es) and e < 0.5, (k, e, es)


def test_model_eval_maps_match_reference_golden(trained_once):
    g = np.load(GOLD)
    emaps = trained_once[3]
    for n, p in zip(("eval_map_x", "eval_map_1", "eval_map_2"), emaps):
        assert GS.rel_max(p, g, n) < 3e-2, (n, GS.rel_max(p, g, n))


def test_transfuse_trainer_eager_and_graph_steps_agree():
    """TransFuseTrainer (multi_train_TransFuse.py:145-197): two optimizer steps, eager vs one captured CUDA graph per step, from the
    same initial state with dropout off: same losses; parameters move; AdamW's first step has the size lr * sign(g) predicts."""
    from mdvit_b200 import ops, synth, transfuse as T
    from mdvit_b200.train_step import TransFuseTrainer
    dev = _dev()
    batches = []
    for d in range(2):
        img, lab = synth.synth_batch(5, d, 2, 256, 256)
        batches.append((img.to(dev), lab.to(torch.uint8).to(dev), d))
    runs = []
    for graph in (False, True):
        torch.manual_seed(0)
        m = T.TransFuse_S_adapt(drop_rate=0.0).to(dev).train()
        ops.manual_seed(7, dev)
        tr = TransFuseTrainer(m, lr=1e-3, weight_decay=0.0)
        p0 = tr.flat.clone()
        if graph:
            tr.capture(batches, warmup=1)
            assert torch.equal(tr.flat, p0)      # capture() restores the training state
            ls = [tr.step_graph(batches).clone() for _ in range(2)]
        else:
            ls = [tr.step(batches).clone() for _ in range(2)]
        torch.cuda.synchronize()
        runs.append((torch.stack(ls).cpu(), tr.flat.clone(), p0))
    (l0, f0, p0), (l1, f1, _) = runs
    assert torch.isfinite(l0).all() and torch.allclose(l0, l1, rtol=2e-3), (l0, l1)
    step1 = (f0 - p0).abs()
    assert step1.max().item() <= 2 * 1e-3 * 1.001 and step1.max().item() > 0.5e-3      # two AdamW steps of at most lr each
    # AdamW's first steps are ~ lr * sign(g): parameters whose true gradient is zero (conv biases in front of a BatchNorm) follow
    # the sign of round-off (fp32 atomics order), so a few elements may differ by up to 2 lr; everything else must agree closely
    diff = (f0 - f1).abs()
    assert diff.median().item() < 5e-5 and (diff > 5e-4).float().mean().item() < 2e-2, (diff.median().item(), (diff > 5e-4).float().mean().item())


def test_stacked_multi_dataset_forward_matches_consecutive_forwards_on_gpu():
    """forward_multi (grouped BatchNorm kernels, one pass over the stack) against one forward per dataset, on the real kernels"""
    from mdvit_b200 import transfuse as T
    dev = _dev()
    img, _, dlab = (t.to(dev) for t in case(B=4))
    outs, bufs = [], []
    for stacked in (True, False):
        torch.manual_seed(0)
        m = T.TransFuse_S_adapt(drop_rate=0.0).to(dev).train()
        with torch.no_grad():
            if stacked:
                maps = m.forward_multi(img, dlab, 2)
            else:
                parts = [m(img[:2], dlab[:2]), m(img[2:], dlab[2:])]
                maps = [torch.cat([a, b]) for a, b in zip(*parts)]
        outs.append(maps)
        bufs.append({k: v.clone() for k, v in m.state_dict().items() if "running" in k or "num_batches" in k})
    for a, b in zip(*outs):
        assert rel(a, b) < 1e-2, rel(a, b)
    for k in bufs[0]:
        assert rel(bufs[0][k], bufs[1][k]) < 1e-2, k


@pytest.mark.parametrize("shape", [(3, 256, 256, 384, 256), (2, 4096, 64, 64, 64), (5, 100, 128, 0, 0), (2, 64, 32, 512, 8)])
def test_gate_cat_fwd_bwd_vs_torch(shape):
    """BiFusion_block's two gates + concat (and Attention_block's x * psi: C2 = C3 = 0) against the torch expression"""
    from mdvit_b200 import ops
    from tests.test_transfuse_wiring import _EmuGateCat
    dev = _dev()
    B, N, C1, C2, C3 = shape
    g = torch.randn(B, N, C1, device=dev).requires_grad_(True)
    p = torch.rand(B, N, 1, device=dev).requires_grad_(True)
    x = torch.randn(B, N, C2, device=dev).requires_grad_(True) if C2 else None
    v = torch.rand(B, C2, device=dev).requires_grad_(True) if C2 else None
    bp = torch.randn(B, N, C3, device=dev).requires_grad_(True) if C3 else None
    probe = torch.randn(B, N, C1 + C2 + C3, device=dev)
    res = []
    for fn in (ops.GateCatFn, _EmuGateCat):
        for t in (g, p, x, v, bp):
            if t is not None:
                t.grad = None
        y = fn.apply(g, p, x, v, bp)
        (y * probe).sum().backward()
        res.append([y.detach()] + [t.grad.clone() for t in (g, p, x, v, bp) if t is not None])
    for a, b in zip(*res):
        assert a.shape == b.shape and rel(a, b) < 1e-5, rel(a, b)


@pytest.mark.parametrize("shape", [(2, 256, 256), (3, 100, 64), (1, 33, 5)])
def test_channel_pool_fwd_bwd_vs_torch(shape):
    from mdvit_b200 import ops
    from tests.test_transfuse_wiring import _EmuChannelPool
    dev = _dev()
    x = torch.randn(*shape, device=dev).requires_grad_(True)
    probe = torch.randn(shape[0], shape[1], 2, device=dev)
    res = []
    for fn in (ops.ChannelPoolFn, _EmuChannelPool):
        x.grad = None
        y = fn.apply(x)
        (y * probe).sum().backward()
        res.append((y.detach(), x.grad.clone()))
    assert torch.equal(res[0][0][..., 0], res[1][0][..., 0]) and rel(res[0][0], res[1][0]) < 1e-6
    assert rel(res[0][1], res[1][1]) < 1e-6


def test_dropout2d_drops_whole_planes_and_backward_reuses_the_mask():
    from mdvit_b200 import ops
    dev = _dev()
    ops.manual_seed(11, dev)
    ops.reset_stream_ids()
    B, N, C, p = 64, 50, 128, 0.2
    x = (torch.rand(B, N, C, device=dev) + 0.5).requires_grad_(True)
    y = ops.Dropout2dFn.apply(x, p)
    ratio = (y / x.detach())                                   # 0 or 1/(1-p), constant over the N pixels of a (sample, channel) plane
    assert torch.allclose(ratio, ratio[:, :1, :].expand_as(ratio))
    plane = ratio[:, 0, :]
    kept = plane > 0
    assert torch.allclose(plane[kept], torch.full_like(plane[kept], 1 / (1 - p)), rtol=1e-6)
    assert abs((~kept).float().mean().item() - p) < 0.02       # 8192 planes: sigma = 0.0044
    y.sum().backward()
    assert torch.allclose(x.grad, ratio)                       # same mask in backward
    y2 = ops.Dropout2dFn.apply(x, p)                           # another call site -> another stream id -> another mask
    assert not torch.equal(y2 > 0, y > 0)


@pytest.mark.parametrize("fused", [False, True])
def test_five_step_trajectory_matches_reference_golden(fused):
    """5 AdamW steps of the reference's training loop (multi_train_TransFuse.py:145-197; oracle/make_golden_transfuse_traj.py ran the
    UNMODIFIED reference): per-step per-dataset losses and the hard Dice of the joint prediction.  The loss falls 1.6 -> 0.58 and
    Dice rises 0.31 -> 0.95 over these steps; at lr 1e-3 the trajectory amplifies operand rounding: the fp32 CPU run with only
    TF32-rounded conv operands and bf16-rounded conv output gradients ends 3-4 % (loss) / 1.6e-2 (Dice) from the reference
    (DESIGN.md section 11), which sets the tolerance here (not the 1e-3 Dice bound MDViT's own trajectory test meets)."""
    from mdvit_b200 import ops, transfuse as T
    from mdvit_b200.train_step import TransFuseTrainer
    from oracle.make_golden_transfuse_traj import LR, STEPS, WD, batches
    dev = _dev()
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "transfuse_traj_golden.npz"))
    torch.manual_seed(0)
    m = T.TransFuse_S_adapt(drop_rate=0.0).to(dev).train()
    tr = TransFuseTrainer(m, lr=LR, weight_decay=WD, fuse_datasets=fused)
    bs = [(i.to(dev), k.to(dev), d) for i, k, d in batches()]
    losses, dice = [], []
    for _ in range(STEPS):
        ls = tr.step(bs)
        losses.append(ls.cpu().numpy())
        dice.append([ops.dice_jaccard(ops.seg_counts(lg, b[1]))[0] for lg, b in zip(tr.last_logits, bs)])
    losses, dice = np.asarray(losses, np.float64), np.asarray(dice, np.float64)
    print("loss rel err per step", np.abs(losses / g["losses"] - 1).max(axis=1), "dice abs err per step", np.abs(dice - g["dice"]).max(axis=1))
    np.testing.assert_allclose(losses[0], g["losses"][0], rtol=2e-3)                 # before any update: the forward alone
    np.testing.assert_allclose(losses, g["losses"], rtol=0.1)                        # measured on the B200: <= 5.1e-2
    assert np.abs(dice - g["dice"]).max() < 6e-2                                     # measured: <= 3.5e-2 (the steep part of the curve)
    assert losses[-1].max() < 0.75 * losses[0].min() and dice[-1].min() > 0.9         # it trains
