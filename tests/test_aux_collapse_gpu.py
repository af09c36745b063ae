"""GPU: the collapsed auxiliary decoder (ops.AuxFn, linear_fuse folded into linear1-4 through the bilinear resize) against
the reference MLPDecoderFM / MLPDecoder under fp32 autograd — logits and every gradient, gradient accumulation, the
da_only backward mode, two backward passes over one graph — and C-ABI tests of its two new kernels in fp64."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from oracle import mdvit_oracle as O

pytestmark = pytest.mark.gpu

BF16_TOL = 1e-2              # logits (measured 2.4-3.5e-3 of abs-max; the concat form measured 4.1-4.9e-3)
# Gradients: bf16 dz through train-mode BatchNorm, whose backward projects out the per-channel mean and the normalised input,
# so every gradient here is a sum with heavy cancellation.  The concat form (one K = 2112 GEMM) measured max-abs / abs-max up
# to 6.1e-2 on the weights and 1.8e-1 on dx1 on these cases, the folded form the same or less.
GRAD_MAX_TOL = 0.25
GRAD_L2_TOL = 5e-2
DIMS = [64, 128, 320, 512]
# Biases whose true gradient is identically zero (a per-channel constant in front of train-mode BatchNorm): compared in
# absolute terms against the scale of the linear_fuse weight gradient (both forms measured up to 1.9e-3 of it).
ZERO_GRAD = ("linear1.bias", "linear2.bias", "linear3.bias", "linear4.bias", "linear_fuse.0.bias")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return torch.device("cuda")


def rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / (b.abs().max() + 1e-30)).item()


def grad_close(a, b):
    a, b = a.double(), b.double()
    return rel(a, b) < GRAD_MAX_TOL and ((a - b).norm() / b.norm()).item() < GRAD_L2_TOL


def make_case(dev, with_x5, B=2, img=256, seed=0):
    from mdvit_b200.model import MLPDecoder, MLPDecoderFM
    torch.manual_seed(seed)
    m = (MLPDecoderFM if with_x5 else MLPDecoder)(DIMS, 1, 512).to(dev).train()
    m.dropout.p = 0.0
    with torch.no_grad():        # non-trivial BatchNorm affine parameters and biases
        bn = m.linear_fuse[1]
        bn.weight.uniform_(0.5, 1.5)
        bn.bias.uniform_(-0.2, 0.2)
        for n, p in m.named_parameters():
            if n.endswith("bias") and "linear_fuse.1" not in n:
                p.uniform_(-0.1, 0.1)
    sizes = [(img // 4 >> i, img // 4 >> i) for i in range(4)]
    g = torch.Generator().manual_seed(seed + 1)
    feats = [torch.randn(B, h * w, c, generator=g).to(dev) for (h, w), c in zip(sizes, DIMS)]
    if with_x5:
        feats.append(torch.randn(B, sizes[0][0] * sizes[0][1], 64, generator=g).to(dev))
    cot = torch.randn(B, 1, img, img, generator=g).to(dev)
    return m, feats, sizes, (img, img), cot


def reference(m, feats, sizes, img_size, cots):
    """fp32 autograd through oracle.mdvit_oracle.mlp_decoder_fm; returns (logits, {param: grad}, [input grads])."""
    sd = {k: (v.detach().double().clone().requires_grad_("running" not in k) if v.is_floating_point() else v.clone())
          for k, v in m.state_dict().items()}
    xs = [f.detach().double().clone().requires_grad_(True) for f in feats]
    B = xs[0].shape[0]
    nchw = [x.transpose(1, 2).reshape(B, x.shape[2], h, w) for x, (h, w) in zip(xs, list(sizes) + [sizes[0]])]
    if len(nchw) == 4:           # MLPDecoder: no main-decoder feature, an empty x5
        nchw.append(nchw[0].new_zeros(B, 0, *sizes[0]))
    out = O.mlp_decoder_fm({"d." + k: v for k, v in sd.items()}, "d", nchw, img_size, training=True, drop2d=0.0)
    tot = sum(cots)
    params = [k for k, v in sd.items() if v.requires_grad]
    grads = torch.autograd.grad(out, [sd[k] for k in params] + xs, tot.double())
    return out.detach(), dict(zip(params, grads[:len(params)])), list(grads[len(params):])


def check_grads(m, gx, ref_g, ref_gx, base=None):
    scale = ref_g["linear_fuse.0.weight"].abs().max().item()
    for n, p in m.named_parameters():
        got = p.grad - (base[n] if base is not None else 0)
        if n in ZERO_GRAD:
            assert (got.double() - ref_g[n]).abs().max().item() < 5e-3 * scale, n
        else:
            assert grad_close(got, ref_g[n]), (n, rel(got, ref_g[n]))
    for i, (a, b) in enumerate(zip(gx, ref_gx)):
        assert grad_close(a, b), (f"dx{i + 1}", rel(a, b))


@pytest.mark.parametrize("with_x5", [True, False])
def test_logits_and_every_gradient_vs_reference(dev, with_x5):
    m, feats, sizes, img_size, cot = make_case(dev, with_x5)
    xs = [f.clone().requires_grad_(True) for f in feats]
    out = m(xs, sizes, img_size)
    ref_out, ref_g, ref_gx = reference(m, feats, sizes, img_size, [cot])
    assert rel(out, ref_out) < BF16_TOL
    out.backward(cot)
    check_grads(m, [x.grad for x in xs], ref_g, ref_gx)


def test_inplace_gradient_targets_accumulate(dev):
    from mdvit_b200 import ops
    m, feats, sizes, img_size, cot = make_case(dev, True, seed=3)
    ops.enable_inplace_grad_accumulation(m.parameters())
    base = {}
    for n, p in m.named_parameters():
        p.grad = torch.randn_like(p)
        base[n] = p.grad.clone()
    xs = [f.clone().requires_grad_(True) for f in feats]
    m(xs, sizes, img_size).backward(cot)
    _, ref_g, ref_gx = reference(m, feats, sizes, img_size, [cot])
    check_grads(m, [x.grad for x in xs], ref_g, ref_gx, base)


def test_da_only_leaves_aux_weight_gradients_untouched(dev):
    from mdvit_b200 import ops
    m, feats, sizes, img_size, cot = make_case(dev, True, seed=4)
    ops.enable_inplace_grad_accumulation(m.parameters())
    base = {}
    for n, p in m.named_parameters():
        p.grad = torch.randn_like(p)
        base[n] = p.grad.clone()
    xs = [f.clone().requires_grad_(True) for f in feats]
    out = m(xs, sizes, img_size)
    with ops.backward_mode("da_only"):
        out.backward(cot)
    for n, p in m.named_parameters():
        assert torch.equal(p.grad, base[n]), n
    _, _, ref_gx = reference(m, feats, sizes, img_size, [cot])
    for i, (x, r) in enumerate(zip(xs, ref_gx)):
        assert grad_close(x.grad, r), (f"dx{i + 1}", rel(x.grad, r))


def test_two_backward_passes_sum(dev):
    m, feats, sizes, img_size, cot = make_case(dev, True, seed=5)
    cot2 = torch.randn_like(cot)
    xs = [f.clone().requires_grad_(True) for f in feats]
    out = m(xs, sizes, img_size)
    out.backward(cot, retain_graph=True)
    out.backward(cot2)
    _, ref_g, ref_gx = reference(m, feats, sizes, img_size, [cot, cot2])
    check_grads(m, [x.grad for x in xs], ref_g, ref_gx)


# ------------------------------------------------------------------------------------------------- C ABI
@pytest.mark.parametrize("B,Ho,Wo,C,ld_out,ins", [
    (2, 64, 64, 512, 512, [(32, 32), (16, 16), (8, 8)]),
    (3, 40, 24, 12, 20, [(17, 9), (5, 31)]),
    (1, 7, 9, 4, 8, [(3, 2)]),
])
def test_upsample_add_matches_interpolate_sum(dev, B, Ho, Wo, C, ld_out, ins):
    from mdvit_b200 import ops
    g = torch.Generator().manual_seed(11)
    out = torch.randn(B * Ho * Wo, ld_out, generator=g).to(dev)
    xs = [(torch.randn(B * h * w, C, generator=g).to(dev), h, w) for h, w in ins]
    ref = out.double().clone()
    for x, h, w in xs:
        up = F.interpolate(x.double().view(B, h, w, C).permute(0, 3, 1, 2), size=(Ho, Wo), mode="bilinear", align_corners=False)
        ref[:, :C] += up.permute(0, 2, 3, 1).reshape(B * Ho * Wo, C)
    ops.upsample_add(out, xs, B, Ho, Wo, C, ld_out=ld_out)
    torch.cuda.synchronize()
    assert (out.double() - ref).abs().max().item() < 1e-5 * ref.abs().max().item()
    assert torch.equal(out[:, C:].double(), ref[:, C:])


MATMUL_CASES = [(512, 512, 64, False, True, True, True), (512, 320, 512, True, False, True, False), (512, 64, 512, False, False, False, False),
                (512, 1, 512, True, False, True, False), (512, 512, 1, False, False, True, True), (37, 53, 70, True, True, False, True),
                (33, 31, 29, False, False, True, False)]


@pytest.mark.parametrize("group", [[c] for c in MATMUL_CASES] + [MATMUL_CASES])
def test_matmul_f32_grouped_matches_fp64(dev, group):
    """Each problem alone and all seven in one launch: transposes, ragged leading dimensions, accumulate, rank-1 addend."""
    from mdvit_b200 import ops
    g = torch.Generator().manual_seed(len(group))
    pad = 3
    probs, checks = [], []
    for M, N, K, ta, tb, acc, uv in group:
        A = torch.randn(K if ta else M, (M if ta else K) + pad, generator=g).to(dev)
        Bm = torch.randn(N if tb else K, (K if tb else N) + pad, generator=g).to(dev)
        C = torch.randn(M, N + pad, generator=g).to(dev)
        u, v = (torch.randn(M, generator=g).to(dev), torch.randn(N, generator=g).to(dev)) if uv else (None, None)
        a = (A[:, :M].t() if ta else A[:, :K]).double()
        b = (Bm[:, :K].t() if tb else Bm[:, :N]).double()
        ref = C.double().clone()
        ref[:, :N] = (ref[:, :N] if acc else 0) + a @ b + (torch.outer(u.double(), v.double()) if uv else 0)
        probs.append(ops.mm(A, Bm, C, M, N, K, lda=A.shape[1], ldb=Bm.shape[1], ldc=C.shape[1], trans_a=ta, trans_b=tb, accumulate=acc,
                            u=u, v=v))
        checks.append((C, ref, N, K))
    ops.matmul_f32(probs)
    torch.cuda.synchronize()
    for C, ref, N, K in checks:
        assert (C.double() - ref).abs().max().item() < 1e-5 * ref.abs().max().item() * max(1.0, K ** 0.5 / 8)
        assert torch.equal(C[:, N:].double(), ref[:, N:])


def test_new_entry_points_reject_bad_arguments(dev):
    from mdvit_b200 import _lib as L
    lib = L.lib()
    assert lib.mdv_matmul_f32_grouped(None, 1, None) == -1
    x = torch.zeros(64, 8, device=dev)
    assert lib.mdv_upsample_add(ctypes.c_void_p(x.data_ptr()), 8, 1, 8, 8, 6, None, 0, 0, None, 0, 0, None, 0, 0, None) == -1
