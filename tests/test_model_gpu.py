"""GPU (B200) model-level parity: the drop-in MDViT module on the sm_100a kernels vs (a) the committed golden vectors
produced by the UNMODIFIED reference (tests/golden, oracle/make_golden.py) and (b) the oracle restatement run in fp32
on the same GPU (TF32 off) on the same seeded inputs.

Tolerances for the bf16 tensor-core path (BASELINE.json north_star asks for "a stated bf16 tolerance, e.g. max relative
error <= 1e-2 on logits"): at 256x256 the logits must agree to relative L2 error <= 2e-2 and max-abs error <= 2e-2 of
the reference abs-max (errors are normalised per tensor as SURVEY.md section 0.8 requires).  Measured: 0.6-1.2e-2 on both
measures with round 1's synthetic weights (2-3e-3 at the reference's random init since the conv trunk runs as TF32,
tests/test_randinit_gpu.py); the only run-to-run spread comes from the atomically accumulated BatchNorm batch sums (fp64)
flipping an occasional bf16 rounding — the attention forward has no atomics and is bit-reproducible; PyTorch's own bf16 autocast of the reference deviates by 2e-2 on the same measure (SURVEY 0.8).  At the tiny 64x64
fixtures the deepest feature map is 2x2 pixels with batch-stat BatchNorm over 8 samples, which amplifies bf16 rounding,
so the fixtures use 3e-2 max-abs.
Gradients: bf16 operands give ~1e-2 relative noise per tensor; tensors whose true gradient is ~0 (biases in front of a
batch-stat BatchNorm) are compared on an absolute scale (relative to the largest gradient in the model).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from mdvit_b200 import synth
from tests.helpers import oracle_state_dict

pytestmark = pytest.mark.gpu

LOGIT_L2_TOL = 2e-2      # ||out - ref||_2 / ||ref||_2
LOGIT_MAX_TOL = 2e-2     # max|out - ref| / max|ref|   (a max over 65k pixels sits ~4 sigma above the rms error)
LOGIT_TOL_64 = 3e-2


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return torch.device("cuda")


def rel(a, b):
    a, b = a.detach().float().cpu(), torch.as_tensor(b).float().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-20)).item()


def rel_l2(a, b):
    a, b = a.detach().double().cpu(), torch.as_tensor(b).double().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def grad_report(grads, ref, loose=("domain_layer", "bridge.")):
    """Per-tensor relative L2 error of the gradients (tensors whose reference gradient is ~0 are measured against the
    largest gradient norm in the model) + the global relative L2 error.  Returns (global, worst_tight, worst_loose, text)."""
    gmax = max(float(torch.as_tensor(r).double().norm()) for r in ref.values() if r is not None)
    rows, num, den = [], 0.0, 0.0
    for n, r in ref.items():
        if r is None or n not in grads:
            continue
        g, r = grads[n].detach().double().cpu(), torch.as_tensor(r).double().cpu()
        e, rn = float((g - r).norm()), float(r.norm())
        num, den = num + e * e, den + rn * rn
        rows.append((e / max(rn, 1e-3 * gmax), n, rn))
    rows.sort(reverse=True)
    tight = [x for x in rows if not any(t in x[1] for t in loose)]
    lo = [x for x in rows if any(t in x[1] for t in loose)]
    text = "; ".join(f"{n}:{e:.3f}" for e, n, _ in rows[:12])
    return (num / den) ** 0.5, (tight[0][0] if tight else 0.0), (lo[0][0] if lo else 0.0), text


def build(dev, img=64, **kw):
    from mdvit_b200.model import MDViT
    m = MDViT(img_size=img, adapt_method="Sup", num_domains=4, decoder_name="MLPFM", **kw).to(dev)
    m.load_state_dict(synth.synth_state_dict(0), strict=True)
    for k in range(1, 5):
        getattr(m, f"debranch{k}").dropout.p = 0.0
    return m


def onehot(d, B, dev):
    return F.one_hot(torch.full((B,), d), 4).float().to(dev)


def test_eval_logits_match_reference_golden_64(dev, golden):
    m = build(dev).eval()
    with torch.no_grad():
        for d in range(4):
            img, _ = synth.synth_batch(1, d, 2, 64, 64)
            out, aux = m(img.to(dev), onehot(d, 2, dev), str(d))
            assert rel(out, golden[f"eval64_out_{d}"]) < LOGIT_TOL_64
            assert rel(aux, golden[f"eval64_aux_{d}"]) < LOGIT_TOL_64


def test_eval_logits_match_reference_golden_256(dev, golden):
    m = build(dev, 256).eval()
    img, _ = synth.synth_batch(2, 3, 1, 256, 256)
    with torch.no_grad():
        out, aux = m(img.to(dev), torch.tensor([[0.0, 0, 0, 1]], device=dev), "3")
    assert out.shape == (1, 1, 256, 256) and aux.shape == (1, 1, 256, 256) and out.dtype == torch.float32
    assert rel_l2(out, golden["eval256_out_3"]) < LOGIT_L2_TOL and rel(out, golden["eval256_out_3"]) < LOGIT_MAX_TOL
    # eval-mode aux logits: the synthetic BN running statistics do not normalise linear_fuse's output, so the 512-term
    # linear_out sum cancels to |aux| ~ 0.02 against a 0.34 abs-max and bf16 operand rounding shows: 4e-2 / 5e-2.
    # (train mode, batch statistics: test_train_logits_256_vs_oracle holds aux to the same 2e-2 as the main logits)
    assert rel_l2(aux, golden["eval256_aux_3"]) < 4e-2 and rel(aux, golden["eval256_aux_3"]) < 5e-2


def test_train_logits_256_vs_oracle(dev):
    """Train-mode forward (BatchNorm batch statistics) at the benchmark resolution against the fp32 oracle on the GPU."""
    from oracle import mdvit_oracle as O
    m = build(dev, 256).train()
    sd = oracle_state_dict(dev)
    img, _ = synth.synth_batch(3, 1, 2, 256, 256)
    img = img.to(dev)
    with torch.no_grad():
        out, aux = m(img, onehot(1, 2, dev), "1")
        ro, ra = O.mdvit_forward(sd, img, onehot(1, 2, dev), "1", training=True)
    assert rel_l2(out, ro) < LOGIT_L2_TOL and rel(out, ro) < LOGIT_MAX_TOL
    assert rel_l2(aux, ra) < LOGIT_L2_TOL and rel(aux, ra) < LOGIT_MAX_TOL
    msd = m.state_dict()
    for k in ("stem.1.bn.running_mean", "bridge.4.running_var", "debranch2.linear_fuse.1.running_var", "decoder4.conv_after.bn.running_mean"):
        assert rel(msd[k], sd[k]) < 5e-3, k


def test_forward_variants_and_dispatch_quirks(dev):
    m = build(dev).eval()
    img, _ = synth.synth_batch(1, 0, 2, 64, 64)
    img = img.to(dev)
    dl = onehot(0, 2, dev)
    with torch.no_grad():
        out, aux = m(img, dl)                       # d=None -> no auxiliary branch (mdvit.py:715-724)
        assert aux is None and out.shape == (2, 1, 64, 64)
        r = m(img, dl, "0", out_feat=True)
        assert set(r) == {"seg", "feat"} and r["feat"].shape == (2, 512)
        r = m(img, dl, out_seg=False)
        assert r["seg"] is None and r["feat"].shape == (2, 512)
        with pytest.raises(TypeError):              # Sup attention needs a label (mdvit.py:350-353)
            m(img, None, "0")
        # mixed-domain batch: the gate is per sample
        dl2 = torch.stack([onehot(0, 1, dev)[0], onehot(3, 1, dev)[0]])
        o2, _ = m(img, dl2)
        o0, _ = m(img, onehot(0, 2, dev))
        o3, _ = m(img, onehot(3, 2, dev))
        # (different BatchNorm-free paths / dropout streams aside, the forward is bit-reproducible: the bound is bf16 rounding noise)
        assert rel_l2(o2[0], o0[0]) < 5e-3 and rel_l2(o2[1], o3[1]) < 5e-3 and rel_l2(o0[1], o3[1]) > 2e-2


@pytest.mark.parametrize("kind", ["MDViT", "MDViT_DSN"])
def test_backward_through_eval_batchnorm_raises(dev, kind):
    """An eval-mode forward with grad enabled records a graph, but its BatchNorms used running statistics (folded into the conv GEMM
    epilogues) and saved nothing to differentiate: backward raises instead of returning gradients of another function."""
    from mdvit_b200.model import MDViT_DSN
    m = build(dev) if kind == "MDViT" else MDViT_DSN(img_size=64, adapt_method="Sup", num_domains=4, decoder_name="MLPFM").to(dev)
    m.eval()
    img, _ = synth.synth_batch(1, 0, 2, 64, 64)
    out, _ = m(img.to(dev), onehot(0, 2, dev), "0")
    assert out.requires_grad
    with pytest.raises(RuntimeError, match="backward through eval-mode BatchNorm is not supported"):
        out.sum().backward()


def _grads_of_step(dev, schedule, fuse_domains=True):
    from mdvit_b200.train_step import MKDTrainer
    m = build(dev).train()
    tr = MKDTrainer(m, schedule=schedule, fuse_domains=fuse_domains)
    batches = [tuple(t.to(dev) for t in synth.synth_batch(1, d, 2, 64, 64)) + (d,) for d in range(4)]
    tr.grad.zero_()
    losses = tr.forward_losses(batches)
    tr.backward(losses)
    torch.cuda.synchronize()
    grads = {n: p.grad.detach().clone() for n, p in m.named_parameters()}
    return m, tr, losses.detach(), grads


def test_train_step_losses_and_gradients_vs_reference_golden(dev, golden):
    m, tr, losses, grads = _grads_of_step(dev, "reference")
    ref_l = golden["train64_losses"]
    assert np.abs(losses.cpu().numpy() - ref_l).max() < 2e-2 * np.abs(ref_l).max()      # per-domain (seg, aux, kt)
    names = [str(n) for n in golden["train64_grad_names"]]
    ref_fp = golden["train64_grad_fp"]
    gmax_norm = ref_fp[:, 0].max()
    dev_norm = sorted((abs(grads[n].double().norm().item() - ref_fp[i, 0]) / max(ref_fp[i, 0], 1e-3 * gmax_norm), n)
                      for i, n in enumerate(names))
    # every gradient tensor's l2 norm is within 10% of the reference's (median within 2%); a 2x2-pixel stage with
    # batch-stat BN over 8 samples (bridge) and the DA's softmax-over-heads cancellation are the noisy ones
    # measured (scripts/dev_margins.py, end of round 2): median 0.0015, worst 0.022 -> bounds at ~3x
    assert dev_norm[len(dev_norm) // 2][0] < 0.005, dev_norm[len(dev_norm) // 2]
    assert all(d < 0.07 for d, n in dev_norm), dev_norm[-8:]
    full = {k.split("/", 1)[1]: golden[k] for k in golden.files if k.startswith("train64_grad/")}
    g_all, w_tight, w_loose, text = grad_report(grads, full)
    assert g_all < 0.02 and w_tight < 0.08 and w_loose < 0.12, text      # measured 0.0074 / 0.032 / 0.044 (scripts/dev_margins.py)
    # BatchNorm running statistics follow nn.BatchNorm2d (momentum 0.1, unbiased running var), 4 forwards
    sd = m.state_dict()
    assert int(sd["stem.0.bn.num_batches_tracked"]) == 4
    assert rel(sd["stem.0.bn.running_var"], golden["train64_bn/stem.0.bn.running_var"]) < 1e-3


def test_single_sweep_schedule_equals_reference_two_pass(dev):
    _, _, l_ref, g_ref = _grads_of_step(dev, "reference")
    _, _, l_one, g_one = _grads_of_step(dev, "single_sweep")
    assert (l_ref - l_one).abs().max().item() < 2e-3 * l_ref.abs().max().item()
    # same math, different bf16 rounding points (one summed cotangent vs two)
    g_all, w_tight, w_loose, text = grad_report(g_one, g_ref)
    assert g_all < 0.02 and w_tight < 0.08 and w_loose < 0.12, text      # measured 0.0074 / 0.032 / 0.044 (scripts/dev_margins.py)


def test_fused_multi_domain_forward_equals_per_domain_forwards(dev):
    """MDViT.forward_multi (one trunk pass over the 4 stacked domain mini-batches, BatchNorm per group) against four
    separate forwards: logits, BatchNorm running statistics, and the gradients of the whole MKD step."""
    m1, m2 = build(dev).train(), build(dev).train()
    batches = [tuple(t.to(dev) for t in synth.synth_batch(1, d, 2, 64, 64)) + (d,) for d in range(4)]
    with torch.no_grad():
        sep = [m1(img, onehot(d, 2, dev), str(d)) for img, _, d in batches]
        x = torch.cat([b[0] for b in batches])
        dl = torch.cat([onehot(d, 2, dev) for _, _, d in batches])
        fused = m2.forward_multi(x, dl, [str(d) for _, _, d in batches])
    for (o1, a1), (o2, a2) in zip(sep, fused):
        assert rel_l2(o2, o1) < 5e-3 and rel_l2(a2, a1) < 1e-2
    sd1, sd2 = m1.state_dict(), m2.state_dict()
    for k in sd1:
        if "running" in k:
            assert rel(sd2[k], sd1[k]) < 5e-3, k
        if k.endswith("num_batches_tracked") and not k.startswith("debranch"):
            assert int(sd1[k]) == int(sd2[k]) == 4, k
    _, _, l_sep, g_sep = _grads_of_step(dev, "single_sweep", fuse_domains=False)
    _, _, l_fus, g_fus = _grads_of_step(dev, "single_sweep", fuse_domains=True)
    assert (l_sep - l_fus).abs().max().item() < 5e-3 * l_sep.abs().max().item()
    g_all, w_tight, w_loose, text = grad_report(g_fus, g_sep)
    assert g_all < 0.02 and w_tight < 0.08 and w_loose < 0.12, text      # measured 0.0074 / 0.032 / 0.044 (scripts/dev_margins.py)


def test_train_step_vs_oracle_on_gpu_and_adamw(dev):
    """Full step incl. fused AdamW against the oracle's autograd + adamw_step on the same device in fp32."""
    from oracle import mdvit_oracle as O
    m, tr, losses, grads = _grads_of_step(dev, "single_sweep")
    sd = oracle_state_dict(dev, requires_grad=True)
    batches = [tuple(t.to(dev) for t in synth.synth_batch(1, d, 2, 64, 64)) + (d,) for d in range(4)]
    Lr, gr = O.train_step_grads(sd, batches)
    ref_l = torch.stack([torch.stack(e) for e in Lr["each"]])
    assert (losses - ref_l).abs().max().item() < 2e-2 * ref_l.abs().max().item()
    g_all, w_tight, w_loose, text = grad_report(grads, {n: gr[n] for n in grads})
    # (against the oracle's fp32 autograd on the GPU the 2x2-pixel bridge / last-stage DA tensors sit at 0.10-0.13, global 0.020)
    assert g_all < 0.03 and w_tight < 0.12 and w_loose < 0.20, text
    # AdamW: p <- p(1 - lr wd) - lr m_hat / (sqrt(v_hat) + eps); at step 1 this is -lr*sign(g) wherever |g| >> eps
    before = {n: p.detach().clone() for n, p in m.named_parameters()}
    tr.optimizer_step()
    torch.cuda.synchronize()
    assert tr.t == 1
    for n, p in m.named_parameters():
        want = before[n].clone()
        O.adamw_step(want, grads[n], torch.zeros_like(want), torch.zeros_like(want), step=1)
        assert (p.detach() - want).abs().max().item() < 1e-6, n


def test_dropout_paths_run_and_are_reproducible(dev):
    """drop_rate / drop_path_rate > 0 (the trainer's setting, multi_train_MDViT.py:59): masks are a pure function of
    (seed, step, stream id), so two identical steps give identical losses and the eval path ignores them."""
    from mdvit_b200 import ops
    from mdvit_b200.model import MDViT
    m = MDViT(img_size=64, drop_rate=0.1, drop_path_rate=0.1, adapt_method="Sup", num_domains=4, decoder_name="MLPFM").to(dev)
    m.load_state_dict(synth.synth_state_dict(0), strict=True)
    m.train()
    img, lab = synth.synth_batch(1, 1, 4, 64, 64)
    img, lab = img.to(dev), lab.to(dev)
    outs = []
    for _ in range(2):
        ops.manual_seed(7, dev)
        ops.reset_stream_ids()
        o, a = m(img, onehot(1, 4, dev), "1")
        l = ops.seg_losses(o, a, lab)
        (l[0] + l[1] + l[2]).backward()
        outs.append(o.detach().clone())
    # identical masks; the second forward sees updated BatchNorm running statistics only in eval mode, but train-mode batch sums are
    # accumulated with (fp64) atomics whose order varies, which can flip a bf16 rounding: close, not necessarily bit-equal
    assert rel(outs[0], outs[1]) < 2e-2 and rel_l2(outs[0], outs[1]) < 5e-3
    assert all(torch.isfinite(p.grad).all().item() for p in m.parameters() if p.grad is not None)
    m.eval()
    with torch.no_grad():
        o1, _ = m(img, onehot(1, 4, dev), "1")
        o2, _ = m(img, onehot(1, 4, dev), "1")
    assert rel_l2(o1, o2) < 5e-3 and rel_l2(o1, outs[0]) > 2e-2


def test_base_logits_match_reference_golden_64(dev, golden):
    """BASE (no DA, no aux branch; BASELINE.json config 2) against logits of the unmodified reference BASE, eval and train mode."""
    from mdvit_b200.model import BASE
    m = BASE(img_size=64, adapt_method=False).to(dev)
    m.load_state_dict(synth.synth_state_dict(0, sup=False, aux=False), strict=True)
    img, _ = synth.synth_batch(4, 0, 2, 64, 64)
    with torch.no_grad():
        assert rel(m.eval()(img.to(dev)), golden["base_eval64_out"]) < LOGIT_TOL_64
        assert rel(m.train()(img.to(dev)), golden["base_train64_out"]) < LOGIT_TOL_64


def test_base_model_without_adapter(dev):
    from mdvit_b200.model import BASE
    from mdvit_b200 import ops
    torch.manual_seed(0)
    m = BASE(img_size=64, adapt_method=False).to(dev).train()
    img, lab = synth.synth_batch(3, 0, 2, 64, 64)
    out = m(img.to(dev))
    assert out.shape == (2, 1, 64, 64)
    l = ops.seg_losses(out, None, lab.to(dev))
    l[0].backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all().item() for p in m.parameters())


def test_base_fused_multi_domain_step_equals_per_domain_step(dev):
    """BASE.forward_multi (one stacked trunk pass, BatchNorm per domain group) through MKDTrainer(with_aux=False) against the
    per-domain loop of multi_train_BASE.py: losses, gradients and BatchNorm running statistics."""
    from mdvit_b200.model import BASE
    from mdvit_b200.train_step import MKDTrainer
    res = {}
    for fuse in (False, True):
        m = BASE(img_size=64, adapt_method=False).to(dev).train()
        m.load_state_dict(synth.synth_state_dict(0, sup=False, aux=False), strict=True)
        tr = MKDTrainer(m, with_aux=False, fuse_domains=fuse)
        batches = [tuple(t.to(dev) for t in synth.synth_batch(1, d, 2, 64, 64)) + (d,) for d in range(4)]
        tr.grad.zero_()
        losses = tr.forward_losses(batches)
        tr.backward(losses)
        torch.cuda.synchronize()
        res[fuse] = (losses.detach().clone(), {n: p.grad.detach().clone() for n, p in m.named_parameters()},
                     {k: v.clone() for k, v in m.state_dict().items() if "running" in k or k.endswith("num_batches_tracked")})
    (l0, g0, b0), (l1, g1, b1) = res[False], res[True]
    assert (l0[:, 0] - l1[:, 0]).abs().max().item() < 5e-3 * l0[:, 0].abs().max().item()
    g_all, w_tight, w_loose, text = grad_report(g1, g0)
    assert g_all < 0.02 and w_tight < 0.08 and w_loose < 0.12, text
    for k in b0:
        if k.endswith("num_batches_tracked"):
            assert int(b0[k]) == int(b1[k]) == 4, k
        else:
            assert rel(b1[k], b0[k]) < 5e-3, k


def test_data_parallel_two_gpus_nccl(dev):
    """One process per GPU over NCCL (skipped on a 1-GPU box): scripts/dp_check.py asserts overlapped == single all-reduce,
    global-batch losses identical on all ranks, replicas in sync after AdamW, and the graph-captured step with NCCL inside."""
    import os
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29533", os.path.join(root, "scripts", "dp_check.py")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.count("DP_OK") == 2, r.stdout[-2000:] + r.stderr[-2000:]


def test_graph_step_keeps_bf16_weight_mirror_fresh(dev):
    """The captured step ends with AdamW followed by ONE launch that re-converts every bf16 GEMM operand copy
    (ops.WeightMirror): after each replay every persistent copy must equal the bf16 cast of the updated fp32 weight, and
    the graph-replayed losses must follow the eager trainer's."""
    from mdvit_b200.train_step import MKDTrainer
    batches = [tuple(t.to(dev) for t in synth.synth_batch(5, d, 2, 64, 64)) + (d,) for d in range(4)]
    m1, m2 = build(dev).train(), build(dev).train()
    eager, graph = MKDTrainer(m1), MKDTrainer(m2)
    before = {k: v.clone() for k, v in m2.state_dict().items()}
    graph.capture(batches, warmup=2)
    # capture() warms up with real optimizer steps but restores parameters, moments, step count and BatchNorm buffers
    assert graph.t == 0 and all(torch.equal(v, before[k]) for k, v in m2.state_dict().items())
    assert float(graph.m.abs().max()) == 0.0 and float(graph.v.abs().max()) == 0.0
    l_eager = [eager.step(batches).clone() for _ in range(2)][-1]
    l_graph = [graph.step_graph(None).clone() for _ in range(2)][-1]
    torch.cuda.synchronize()
    assert graph.t == 2 and eager.t == 2
    checked = 0
    for (_, mode, _), (ref, _, dst, rows, cols, out_ld, _, cin) in graph.mirror.entries.items():
        w = ref()
        if mode == 0:
            assert torch.equal(dst[:, :cols], w.detach().reshape(rows, cols).bfloat16()), "stale bf16 copy"
            checked += 1
        elif mode == 1:
            assert torch.equal(dst[:, :rows], w.detach().reshape(rows, cols).t().bfloat16()), "stale transposed bf16 copy"
            checked += 1
    assert checked > 100
    assert (l_eager - l_graph).abs().max().item() < 2e-2 * l_eager.abs().max().item()
