"""MDViT_DSN (domain-specific norms; SURVEY.md section 8f-3; Models/Transformer/mdvit.py:735-960): schema and random init on
CPU, logits against golden outputs of the UNMODIFIED reference on the GPU (oracle/make_golden_dsn.py)."""
import os

import numpy as np
import pytest
import torch

from mdvit_b200 import synth
from oracle.golden_sample import rel_max
from tests.helpers import fingerprint

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def dgold():
    return np.load(os.path.join(ROOT, "tests", "golden", "mdvit_dsn_golden.npz"), allow_pickle=False)


def build():
    from mdvit_b200.model import MDViT_DSN
    torch.manual_seed(0)
    return MDViT_DSN(img_size=64, adapt_method="Sup", num_domains=4, decoder_name="MLPFM")


def test_dsn_state_dict_schema_and_random_init_match_the_reference(dgold):
    m = build()
    assert list(m.state_dict().keys()) == [str(k) for k in dgold["keys"]] and len(dgold["keys"]) == 980
    fp = fingerprint(list(m.named_parameters()))
    assert np.abs(fp - dgold["init_fp"]).max() <= 1e-9 * np.abs(dgold["init_fp"]).max()
    from mdvit_b200.model import MDViT, MDViT_DSN
    assert len(MDViT_DSN(img_size=64, adapt_method="Sup").state_dict()) == 980     # the reference default decoder_name is "MLP"
    with pytest.raises(NotImplementedError):
        MDViT_DSN(img_size=64, decoder_name="DeepLabV3")
    with pytest.raises(NotImplementedError):
        MDViT_DSN(img_size=64, decoder_name="Transformer")
    assert list(MDViT(img_size=64, adapt_method="Sup", decoder_name="MLP").state_dict().keys()) == [str(k) for k in dgold["mlp_keys"]]


@pytest.mark.gpu
def test_dsn_logits_match_reference_golden(dgold):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    dev = torch.device("cuda")
    m = build()
    m.load_state_dict(synth.dsn_perturb(m.state_dict()), strict=True)
    for k in range(1, 5):
        getattr(m, f"debranch{k}").dropout.p = 0.0
    m = m.to(dev)

    def rel(a, b):
        b = torch.as_tensor(b)
        return ((a.detach().float().cpu() - b).abs().max() / b.abs().max()).item()

    outs = {}
    with torch.no_grad():
        for mode in ("eval", "train"):
            m.train(mode == "train")
            for d in (1, 3):
                img, _ = synth.synth_batch(11, d, 2, 64, 64)
                dl = torch.nn.functional.one_hot(torch.full((2,), d), 4).float().to(dev)
                o, a = m(img.to(dev), dl, str(d))
                outs[(mode, d)] = o
                assert rel(o, dgold[f"{mode}_out_{d}"]) < 2e-2 and rel(a, dgold[f"{mode}_aux_{d}"]) < 2e-2, (mode, d)
        # the domain index selects the norm set: same image, other d -> different logits
        m.eval()
        img, _ = synth.synth_batch(11, 1, 2, 64, 64)
        dl = torch.nn.functional.one_hot(torch.full((2,), 1), 4).float().to(dev)
        o_other = m(img.to(dev), dl, "2")[0]
        assert rel(o_other, outs[("eval", 1)].cpu()) > 5e-2
    with pytest.raises((TypeError, ValueError)):
        m(img.to(dev), dl, None)          # int(d) is required by the reference as well


def test_transformer_aux_decoder_schema_and_random_init_match_the_reference(dgold):
    """decoder_name='Transformer' (mdvit.py:613-642; SURVEY.md section 8f-4): 1460 state_dict keys, bit-identical init."""
    from mdvit_b200.model import MDViT
    torch.manual_seed(0)
    m = MDViT(img_size=64, adapt_method="Sup", num_domains=4, decoder_name="Transformer")
    assert list(m.state_dict().keys()) == [str(k) for k in dgold["tr_keys"]] and len(dgold["tr_keys"]) == 1460
    fp = fingerprint(list(m.named_parameters()))
    assert np.abs(fp - dgold["tr_init_fp"]).max() <= 1e-9 * np.abs(dgold["tr_init_fp"]).max()


@pytest.mark.gpu
def test_transformer_aux_decoder_logits_match_reference_golden(dgold):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from mdvit_b200 import ops
    from mdvit_b200.model import MDViT
    from oracle.make_golden_dsn import aux_state
    dev = torch.device("cuda")
    m = MDViT(img_size=64, adapt_method="Sup", num_domains=4, decoder_name="Transformer")
    m.load_state_dict(synth.synth_state_dict(0, aux=False) | aux_state(m, "debranchs"), strict=True)
    m = m.to(dev)

    def rel(a, b):
        b = torch.as_tensor(b)
        return ((a.detach().float().cpu() - b).abs().max() / b.abs().max()).item()

    for mode in ("eval", "train"):
        m.train(mode == "train")
        for d in (0, 3):
            img, lab = synth.synth_batch(14, d, 2, 64, 64)
            dl = torch.nn.functional.one_hot(torch.full((2,), d), 4).float().to(dev)
            with torch.no_grad():
                o, a = m(img.to(dev), dl, str(d))
            # (the auxiliary logits are small here — abs-max ~1.2 after 8 more bf16 blocks — so max-abs/abs-max is the noisier
            # figure; the error is a smooth offset of ~1e-2 absolute, the same size as the main output's: bound both ratios at 4e-2)
            assert rel(o, dgold[f"tr_{mode}_out_{d}"]) < 2e-2 and rel(a, dgold[f"tr_{mode}_aux_{d}"]) < 4e-2, (mode, d)
            ra = torch.as_tensor(dgold[f"tr_{mode}_aux_{d}"])
            assert ((a.float().cpu() - ra).norm() / ra.norm()).item() < 4e-2, (mode, d)
    # the stacked multi-domain forward gives the same auxiliary logits as the per-domain calls (eval: no batch statistics;
    # the train-mode forwards above moved the BatchNorm running statistics: restore them first)
    m.load_state_dict({k: v.to(dev) for k, v in (synth.synth_state_dict(0, aux=False) | aux_state(m, "debranchs")).items()}, strict=True)
    m.eval()
    imgs = torch.cat([synth.synth_batch(14, d, 2, 64, 64)[0] for d in (0, 3)]).to(dev)
    dls = torch.cat([torch.nn.functional.one_hot(torch.full((2,), d), 4).float() for d in (0, 3)]).to(dev)
    with torch.no_grad():
        res = m.forward_multi(imgs, dls, ["0", "3"])
    for (o, a), d in zip(res, (0, 3)):
        assert rel(o, dgold[f"tr_eval_out_{d}"]) < 2e-2 and rel(a, dgold[f"tr_eval_aux_{d}"]) < 4e-2
    # and it trains: only the selected domain's decoder receives gradients
    m.train()
    o, a = m(img.to(dev), dl, "3")
    ops.seg_losses(o, a, lab.to(dev)).sum().backward()
    g3 = [p.grad for n, p in m.named_parameters() if n.startswith("debranchs.3.")]
    assert all(g is not None and torch.isfinite(g).all().item() for g in g3)
    assert all(p.grad is None or p.grad.abs().max().item() == 0 for n, p in m.named_parameters() if n.startswith("debranchs.0."))
    with pytest.raises((TypeError, ValueError)):
        m(img.to(dev), dl, None)


def test_deeplab_aux_decoder_schema_and_random_init_match_the_reference(dgold):
    """decoder_name='DeepLabV3' (mdvit.py:608-611, Decoders.py:218-235): 716 state_dict keys, bit-identical init."""
    from mdvit_b200.model import MDViT
    torch.manual_seed(0)
    m = MDViT(img_size=256, adapt_method="Sup", num_domains=4, decoder_name="DeepLabV3")
    assert list(m.state_dict().keys()) == [str(k) for k in dgold["dl_keys"]] and len(dgold["dl_keys"]) == 716
    fp = fingerprint(list(m.named_parameters()))
    assert np.abs(fp - dgold["dl_init_fp"]).max() <= 1e-9 * np.abs(dgold["dl_init_fp"]).max()
    with pytest.raises(NotImplementedError):
        MDViT(img_size=64, decoder_name="UNet")


@pytest.mark.gpu
def test_deeplab_aux_decoder_logits_and_gradients_match_reference_golden(dgold):
    """ASPP with dilated 3x3 convs on the 8x8 encoder map (256x256 input), image pooling, project, 3x3 conv, head: logits in eval
    and train mode and the gradients of sum(aux * R) (branch parameters + the stem, i.e. through the decoder's input gradient)."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from mdvit_b200.model import MDViT
    from oracle.make_golden_dsn import aux_state
    dev = torch.device("cuda")
    m = MDViT(img_size=256, adapt_method="Sup", num_domains=4, decoder_name="DeepLabV3")
    m.load_state_dict(synth.synth_state_dict(0, aux=False) | aux_state(m, "debranch"), strict=True)
    for k in range(1, 5):
        getattr(m, f"debranch{k}").classifier[0].project[3].p = 0.0
    m = m.to(dev)
    img, _ = synth.synth_batch(15, 1, 2, 256, 256)
    dl = torch.nn.functional.one_hot(torch.full((2,), 1), 4).float().to(dev)

    m.eval()
    with torch.no_grad():
        o, a = m(img.to(dev), dl, "1")
    assert rel_max(o, dgold, "dl_eval_out") < 2e-2 and rel_max(a, dgold, "dl_eval_aux") < 3e-2
    m.train()
    o, a = m(img.to(dev), dl, "1")
    assert rel_max(a, dgold, "dl_train_aux") < 3e-2
    R = synth.synth_tensor("dl_probe", tuple(a.shape)).to(dev)
    (a * R).sum().backward()
    names = [str(n) for n in dgold["dl_grad_names"]]
    params = dict(m.named_parameters())
    fp = fingerprint([(n, params[n].grad) for n in names])
    ref = dgold["dl_grad_fp"]
    bad = []
    for i, n in enumerate(names):
        # Only 2 x 8 x 8 = 128 rows feed every BatchNorm / ReLU of the decoder here, so a handful of ReLU masks flipped by the bf16
        # forward moves a gradient by several percent: norms within 8 %, probe projections within 0.4 of the norm.  The tight
        # check of the backward is test_deeplab_fn_matches_stock_pytorch_modules (same op in torch fp32, more rows, cosines).
        if abs(fp[i, 0] - ref[i, 0]) > 0.08 * ref[i, 0] + 1e-6 or abs(fp[i, 1] - ref[i, 1]) > 0.40 * ref[i, 0] + 1e-6:
            bad.append((n, fp[i].tolist(), ref[i].tolist()))
    assert not bad, bad[:6]
    assert all(params[n].grad is None or params[n].grad.abs().max().item() == 0 for n in params if n.startswith("debranch1."))
    # dropout on: runs, finite, and the mask is the same in forward and backward (gradient of a linear probe is reproducible)
    m.debranch2.classifier[0].project[3].p = 0.1
    m.zero_grad()
    o, a = m(img.to(dev), dl, "1")
    (a * R).sum().backward()
    assert torch.isfinite(a).all().item() and all(torch.isfinite(params[n].grad).all().item() for n in names)


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,W", [(8, 8, 8), (3, 7, 10)])
def test_deeplab_fn_matches_stock_pytorch_modules(B, H, W):
    """ops.DeepLabFn + HeadFn against the SAME decoder evaluated by stock PyTorch (its parameter containers are plain
    nn.Conv2d / BatchNorm2d / ReLU Sequentials with the reference's structure, so `classifier(x)` is the reference arithmetic in
    fp32): outputs, input gradient and every parameter gradient, train mode (batch statistics), dropout off."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import copy
    from mdvit_b200.model import DeepLabV3Decoder
    dev = torch.device("cuda")
    torch.manual_seed(3)
    dec = DeepLabV3Decoder(512, 1)
    with torch.no_grad():
        for n, p in dec.named_parameters():      # BN affine parameters away from (1, 0)
            if p.dim() == 1 and "classifier.4" not in n:
                p.copy_(1.0 + 0.2 * torch.randn_like(p) if n.endswith("weight") else 0.2 * torch.randn_like(p))
    dec.classifier[0].project[3].p = 0.0
    dec = dec.to(dev).train()
    ref = copy.deepcopy(dec)
    x = torch.randn(B, H * W, 512, device=dev)
    probe = torch.randn(B, 1, 32 * H, 32 * W, device=dev)
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        xr = x.clone().requires_grad_(True)
        F = torch.nn.functional
        aspp = ref.classifier[0]            # Utils/_deeplab.py:137-165 with stock torch ops (the containers carry no forward)
        xn = xr.transpose(1, 2).reshape(B, 512, H, W)
        res = [aspp.convs[k](xn) for k in range(4)]
        res.append(F.interpolate(aspp.convs[4](xn), size=(H, W), mode="bilinear", align_corners=False))
        t = aspp.project(torch.cat(res, dim=1))
        for layer in list(ref.classifier)[1:]:
            t = layer(t)
        yr = F.interpolate(t, size=(32 * H, 32 * W), mode="bilinear", align_corners=False)
        (yr * probe).sum().backward()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    xo = x.clone().requires_grad_(True)
    feats = [None, None, None, xo]
    yo = dec(feats, [None, None, None, (H, W)], (32 * H, 32 * W))
    (yo * probe).sum().backward()

    def cos(a, b):
        a, b = a.flatten().double(), b.flatten().double()
        return (a @ b / (a.norm() * b.norm() + 1e-30)).item()

    assert ((yo - yr).abs().max() / yr.abs().max()).item() < 2e-2
    assert cos(xo.grad, xr.grad) > 0.99 and abs(xo.grad.norm().item() / xr.grad.norm().item() - 1) < 0.03      # (bf16 operands, a few hundred rows)
    worst = min((cos(p.grad, q.grad), n) for (n, p), (_, q) in zip(dec.named_parameters(), ref.named_parameters()))
    assert worst[0] > 0.99, worst
    for (n, p), (_, q) in zip(dec.named_parameters(), ref.named_parameters()):
        assert abs(p.grad.norm().item() / (q.grad.norm().item() + 1e-30) - 1) < 0.05, n
    # running statistics advanced identically (train-mode BatchNorm side effect)
    for (n, b1), (_, b2) in zip(dec.named_buffers(), ref.named_buffers()):
        if b1.is_floating_point():
            assert (b1 - b2).abs().max().item() <= 2e-2 * (b2.abs().max().item() + 1e-3), n
        else:
            assert torch.equal(b1, b2), n


@pytest.mark.parametrize("am", ["Sup", None])
def test_base_dsn_schema_and_random_init_match_the_reference(dgold, am):
    """BASE_DSN (base.py:515-696; SURVEY.md section 8f-3): 912 / 848 state_dict keys, bit-identical stock-constructor init."""
    from mdvit_b200.model import BASE_DSN
    tag = "sup" if am else "plain"
    torch.manual_seed(0)
    m = BASE_DSN(img_size=64, adapt_method=am, num_domains=4)
    assert list(m.state_dict().keys()) == [str(k) for k in dgold[f"base_dsn_{tag}_keys"]]
    fp = fingerprint(list(m.named_parameters()))
    ref = dgold[f"base_dsn_{tag}_init_fp"]
    assert np.abs(fp - ref).max() <= 1e-9 * np.abs(ref).max()


@pytest.mark.gpu
@pytest.mark.parametrize("am", ["Sup", None])
def test_base_dsn_logits_match_reference_golden(dgold, am):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from mdvit_b200.model import BASE_DSN
    dev = torch.device("cuda")
    tag = "sup" if am else "plain"
    torch.manual_seed(0)
    m = BASE_DSN(img_size=64, adapt_method=am, num_domains=4)
    m.load_state_dict(synth.dsn_perturb(m.state_dict()), strict=True)
    m = m.to(dev)
    with torch.no_grad():
        for mode in ("eval", "train"):
            m.train(mode == "train")
            for d in (0, 2):
                img, _ = synth.synth_batch(13, d, 2, 64, 64)
                dl = torch.nn.functional.one_hot(torch.full((2,), d), 4).float().to(dev) if am else None
                o = m(img.to(dev), dl, str(d))
                ref = torch.as_tensor(dgold[f"base_dsn_{tag}_{mode}_{d}"])
                assert tuple(o.shape) == tuple(ref.shape)
                assert ((o.float().cpu() - ref).abs().max() / ref.abs().max()).item() < 2e-2, (mode, d)
        m.eval()
        f = m(img.to(dev), dl, "2", out_feat=True)
        assert tuple(f["feat"].shape) == (2, 512) and tuple(f["seg"].shape) == (2, 1, 64, 64)
        assert m(img.to(dev), dl, "2", out_seg=False)["seg"] is None


@pytest.mark.gpu
def test_mlp_aux_decoder_logits_match_reference_golden(dgold):
    """decoder_name='MLP' (Decoders.MLPDecoder: MLPDecoderFM without the main-decoder feature) against the unmodified reference."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from mdvit_b200.model import MDViT
    from oracle.make_golden_dsn import mlp_aux_state
    dev = torch.device("cuda")
    m = MDViT(img_size=64, adapt_method="Sup", num_domains=4, decoder_name="MLP")
    m.load_state_dict(synth.synth_state_dict(0, aux=False) | mlp_aux_state(m), strict=True)
    for k in range(1, 5):
        getattr(m, f"debranch{k}").dropout.p = 0.0
    m = m.to(dev)
    img, lab = synth.synth_batch(12, 2, 2, 64, 64)
    dl = torch.nn.functional.one_hot(torch.full((2,), 2), 4).float().to(dev)
    for mode in ("eval", "train"):
        m.train(mode == "train")
        with torch.no_grad():
            o, a = m(img.to(dev), dl, "2")
        for t, ref in ((o, dgold[f"mlp_{mode}_out"]), (a, dgold[f"mlp_{mode}_aux"])):
            ref = torch.as_tensor(ref)
            assert ((t.float().cpu() - ref).abs().max() / ref.abs().max()).item() < 3e-2, mode
    # and it trains: the MKD losses back-propagate through the 2048-channel fuse
    from mdvit_b200 import ops
    m.train()
    o, a = m(img.to(dev), dl, "2")
    ops.seg_losses(o, a, lab.to(dev)).sum().backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all().item() for n, p in m.named_parameters() if "debranch3" in n or "stem" in n)
