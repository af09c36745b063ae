"""softmax(QK^T)V attention with the DA head gate (TransFuse_S_adapt's DeiT-S branch, BASELINE.json config 4 / SURVEY 8f-1):
 * CPU: the oracle restatement (oracle.mdvit_oracle.attention_sup) against golden outputs of the UNMODIFIED reference
   Attention_Sup / Attention modules (oracle/make_golden_transfuse.py);
 * GPU: qkv GEMM -> mdv_da_gate_fwd -> mdv_sdpa_fwd (tcgen05) -> proj GEMM through the C ABI against the same goldens.
Tolerance of the bf16 tensor-core path: 1e-2 of the tensor abs-max (bf16 q/k/v, bf16 probabilities, fp32 accumulation)."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle.golden_sample import rel_l2, rel_max
from oracle.make_golden_transfuse import DIM, HEADS, N, attention_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def tgold():
    return np.load(os.path.join(ROOT, "tests", "golden", "transfuse_attention_golden.npz"), allow_pickle=False)


def rel(a, b):
    a, b = torch.as_tensor(a).float().cpu(), torch.as_tensor(b).float().cpu()
    return ((a - b).abs().max() / b.abs().max()).item()


def test_oracle_attention_sup_matches_reference_golden(tgold):
    from oracle import mdvit_oracle as O
    sd, x, label = attention_case()
    sd = {"a." + k: v for k, v in sd.items()}
    out, pre = O.attention_sup(sd, "a", x, label, HEADS, return_pre_proj=True)
    assert rel_max(out, tgold, "sup_out") < 2e-3 and rel_max(pre, tgold, "sup_pre_proj") < 2e-3   # fp16 storage
    out2, pre2 = O.attention_sup(sd, "a", x, None, HEADS, return_pre_proj=True)
    assert rel_max(out2, tgold, "plain_out") < 2e-3 and rel_max(pre2, tgold, "plain_pre_proj") < 2e-3


@pytest.mark.gpu
@pytest.mark.parametrize("sup", [True, False])
def test_sdpa_kernel_matches_reference_attention_golden(tgold, sup):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from mdvit_b200 import _lib as L
    lib, dev = L.lib(), torch.device("cuda")
    sd, x, label = attention_case()
    sd = {k: v.to(dev) for k, v in sd.items()}
    B, M = x.shape[0], x.shape[0] * N
    xb = x.to(dev).reshape(M, DIM).bfloat16()
    qkv = torch.empty(M, 3 * DIM, device=dev, dtype=torch.bfloat16)
    e = L.GemmEpi()
    e.out, e.ldc, e.out_bf16, e.bias = L.ptr(qkv), 3 * DIM, 1, L.ptr(sd["qkv.bias"])
    wq = sd["qkv.weight"].bfloat16()
    L.check(lib.mdv_gemm_nt(L.ptr(xb), DIM, L.ptr(wq), DIM, M, 3 * DIM, DIM, ctypes.byref(e), L.stream()), "qkv")
    gate = None
    if sup:
        hid = sd["domain_layer.0.weight"].shape[0]
        gate, hidb = torch.empty(B, DIM, device=dev), torch.empty(B, hid, device=dev)
        lab = label.to(dev)
        L.check(lib.mdv_da_gate_fwd(L.ptr(lab), L.ptr(sd["domain_layer.0.weight"]), L.ptr(sd["domain_layer.0.bias"]), L.ptr(sd["domain_layer.2.weight"]),
                                    L.ptr(sd["domain_layer.2.bias"]), L.ptr(hidb), L.ptr(gate), B, 4, hid, DIM, HEADS, L.stream()), "gate")
    y = torch.empty(M, DIM, device=dev, dtype=torch.bfloat16)
    lse = torch.empty(B, HEADS, N, device=dev)
    L.check(lib.mdv_sdpa_fwd(L.ptr(qkv), L.ptr(gate), L.ptr(y), L.ptr(lse), B, N, DIM, HEADS, ctypes.c_float((DIM // HEADS) ** -0.5), L.stream()), "sdpa")
    out = torch.empty(M, DIM, device=dev)
    e2 = L.GemmEpi()
    e2.out, e2.ldc, e2.out_bf16, e2.bias = L.ptr(out), DIM, 0, L.ptr(sd["proj.bias"])
    wp = sd["proj.weight"].bfloat16()
    L.check(lib.mdv_gemm_nt(L.ptr(y), DIM, L.ptr(wp), DIM, M, DIM, DIM, ctypes.byref(e2), L.stream()), "proj")
    key = "sup" if sup else "plain"
    assert rel_max(y.reshape(B, N, DIM), tgold, key + "_pre_proj") < 1e-2
    assert rel_max(out.reshape(B, N, DIM), tgold, key + "_out") < 1e-2
    # the saved log-sum-exp is that of the scaled scores
    q, k = qkv.float().reshape(B, N, 3, HEADS, 64)[:, :, 0], qkv.float().reshape(B, N, 3, HEADS, 64)[:, :, 1]
    s = torch.einsum("bnhd,bmhd->bhnm", q, k) * 0.125
    assert rel(lse, torch.logsumexp(s, dim=-1)) < 2e-3
    # N = 128 variant and odd batch: against torch on the same bf16 qkv
    for Bn, Nn in ((3, 128), (5, 256)):
        torch.manual_seed(Bn)
        qkv2 = (torch.randn(Bn * Nn, 3 * DIM, device=dev) * 1.5).bfloat16()
        g2 = torch.softmax(torch.randn(Bn, HEADS, 64, device=dev), dim=1).reshape(Bn, DIM).contiguous() if sup else None
        y2 = torch.empty(Bn * Nn, DIM, device=dev, dtype=torch.bfloat16)
        L.check(lib.mdv_sdpa_fwd(L.ptr(qkv2), L.ptr(g2), L.ptr(y2), None, Bn, Nn, DIM, HEADS, ctypes.c_float(0.125), L.stream()), "sdpa")
        t = qkv2.float().reshape(Bn, Nn, 3, HEADS, 64)
        a = torch.softmax(torch.einsum("bnhd,bmhd->bhnm", t[:, :, 0], t[:, :, 1]) * 0.125, dim=-1)
        ref = torch.einsum("bhnm,bmhd->bnhd", a, t[:, :, 2])
        if sup:
            ref = ref * g2.reshape(Bn, 1, HEADS, 64)
        assert rel(y2.reshape(Bn, Nn, HEADS, 64), ref) < 1e-2


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,heads,sup", [(2, 256, 6, True), (3, 128, 2, False), (1, 256, 1, True)])
def test_sdpa_backward_matches_torch_autograd(B, N, heads, sup):
    """mdv_sdpa_bwd (mma.sync, P recomputed from the log-sum-exp) against torch autograd of the same op in fp32 on the same
    bf16-rounded q, k, v and output gradient: dq, dk, dv within 2e-2 of each tensor's abs-max (bf16 P / dS operands, bf16
    outputs), the gate gradient within 1e-2."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from mdvit_b200 import _lib as L
    lib, dev = L.lib(), torch.device("cuda")
    torch.manual_seed(5)
    C = heads * 64
    scale = 64 ** -0.5
    qkv = (torch.randn(B, N, 3 * C, device=dev) * 1.5).bfloat16()
    gate = torch.softmax(torch.randn(B, heads, 64, device=dev), dim=1).reshape(B, C).contiguous() if sup else None
    dy = torch.randn(B, N, C, device=dev).bfloat16()
    out = torch.empty(B, N, C, device=dev, dtype=torch.bfloat16)
    lse = torch.empty(B, heads, N, device=dev)
    st = L.stream()
    L.check(lib.mdv_sdpa_fwd(L.ptr(qkv), L.ptr(gate), L.ptr(out), L.ptr(lse), B, N, C, heads, ctypes.c_float(scale), st), "sdpa_fwd")
    dqkv = torch.full((B, N, 3 * C), float("nan"), device=dev, dtype=torch.bfloat16)
    dgate = torch.full((B, C), float("nan"), device=dev) if sup else None
    L.check(lib.mdv_sdpa_bwd(L.ptr(qkv), L.ptr(gate), L.ptr(out), L.ptr(lse), L.ptr(dy), L.ptr(dqkv), L.ptr(dgate), B, N, C, heads,
                             ctypes.c_float(scale), st), "sdpa_bwd")
    # reference: fp32 autograd
    x = qkv.float().requires_grad_(True)
    gr = gate.clone().requires_grad_(True) if sup else None
    q, k, v = (t.reshape(B, N, heads, 64).transpose(1, 2) for t in x.split(C, dim=2))
    p = torch.softmax((q @ k.transpose(-1, -2)) * scale, dim=-1)
    y = (p @ v).transpose(1, 2).reshape(B, N, C)
    if sup:
        y = y * gr[:, None, :]
    assert ((out.float() - y).abs().max() / y.abs().max()).item() < 1e-2
    y.backward(dy.float())
    for name, sl in (("dq", slice(0, C)), ("dk", slice(C, 2 * C)), ("dv", slice(2 * C, 3 * C))):
        a, r = dqkv[:, :, sl].float(), x.grad[:, :, sl]
        assert torch.isfinite(a).all().item(), name
        assert ((a - r).abs().max() / r.abs().max()).item() < 2e-2, (name, ((a - r).abs().max() / r.abs().max()).item())
        assert ((a - r).norm() / r.norm()).item() < 1.5e-2, name
    if sup:
        assert ((dgate - gr.grad).abs().max() / gr.grad.abs().max()).item() < 1e-2


@pytest.mark.gpu
@pytest.mark.parametrize("sup", [True, False])
def test_attention_module_dropin_forward_backward_match_reference(tgold, sup):
    """mdvit_b200.transfuse.Attention_Sup / Attention (same ctor / state_dict / forward as vision_transformer.py:96-169): output,
    input gradient and every parameter gradient of sum(y * R) against the unmodified reference modules."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from mdvit_b200 import transfuse as T
    from oracle.make_golden_transfuse import _t, grad_sample
    dev = torch.device("cuda")
    sd, x, label = attention_case()
    key = "sup" if sup else "plain"
    if sup:
        m = T.Attention_Sup(DIM, num_heads=HEADS, qkv_bias=True)
        m.load_state_dict(sd, strict=True)
    else:
        m = T.Attention(DIM, num_heads=HEADS, qkv_bias=True)
        m.load_state_dict({k: v for k, v in sd.items() if not k.startswith("domain_layer")}, strict=True)
    m = m.to(dev).train()
    xr = x.to(dev).requires_grad_(True)
    y = m(xr, label.to(dev)) if sup else m(xr)
    assert rel_max(y, tgold, key + "_out") < 1e-2
    R = _t("tfprobe", tuple(y.shape), 1.0).to(dev)
    (y * R).sum().backward()
    assert rel_max(xr.grad, tgold, key + "_dx") < 2e-2
    for n, p in m.named_parameters():
        err = rel_l2(grad_sample(p.grad), tgold, f"{key}_grad.{n}")
        assert err < 2e-2, (n, err)
    with pytest.raises(NotImplementedError):
        T.Attention(256, num_heads=8)          # head_dim 32


def test_deit_adapt_schema_and_random_init_match_the_reference(tgold):
    """deit_small_patch16_224_adapt (DeiT.py:157-181): 134 state_dict keys, bit-identical stock-constructor init, pos_embed [1,256,384]."""
    from mdvit_b200.transfuse import deit_small_patch16_224_adapt
    from tests.helpers import fingerprint
    torch.manual_seed(0)
    m = deit_small_patch16_224_adapt(pretrained=False, num_domains=4)
    assert list(m.state_dict().keys()) == [str(k) for k in tgold["deit_keys"]] and tuple(m.pos_embed.shape) == (1, 256, 384)
    fp = fingerprint(list(m.named_parameters()))
    assert np.abs(fp - tgold["deit_init_fp"]).max() <= 1e-9 * np.abs(tgold["deit_init_fp"]).max()


@pytest.mark.gpu
def test_deit_adapt_tokens_and_gradients_match_reference(tgold):
    """The transformer branch of TransFuse_S_adapt end to end (patch embedding GEMM + pos_embed, 8 Block_adapt, final LayerNorm) at the
    reference's own random init: output tokens and the gradients of a probe loss for all 133 trained parameters."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from mdvit_b200.transfuse import deit_small_patch16_224_adapt
    from oracle.make_golden_transfuse import _t
    from tests.helpers import fingerprint
    dev = torch.device("cuda")
    torch.manual_seed(0)
    m = deit_small_patch16_224_adapt(pretrained=False, num_domains=4)
    with torch.no_grad():
        m.pos_embed.copy_(_t("deitpos", tuple(m.pos_embed.shape), 0.02))
    m = m.to(dev).train()
    img = _t("deitimg", (2, 3, 256, 256), 1.0).to(dev)
    dlab = torch.nn.functional.one_hot(torch.tensor([1, 3]), 4).float().to(dev)
    tok = m(img, dlab)
    assert rel_max(tok, tgold, "deit_tokens") < 1e-2
    Rd = _t("deitprobe", tuple(tok.shape), 1.0).to(dev)
    (tok * Rd).sum().backward()
    names = [str(n) for n in tgold["deit_grad_names"]]
    P = dict(m.named_parameters())
    assert set(names) == {n for n, p in P.items() if p.grad is not None}
    fp, ref = fingerprint([(n, P[n].grad) for n in names]), tgold["deit_grad_fp"]
    bad = [(n, fp[i].tolist(), ref[i].tolist()) for i, n in enumerate(names)
           if abs(fp[i, 0] - ref[i, 0]) > 0.03 * ref[i, 0] + 1e-7 or abs(fp[i, 1] - ref[i, 1]) > 0.06 * ref[i, 0] + 1e-7]
    assert not bad, bad[:5]
    for n in names:
        if "deit_grad." + n in tgold.files:
            e = rel_l2(P[n].grad, tgold, "deit_grad." + n)
            assert e < 3e-2, (n, e)
