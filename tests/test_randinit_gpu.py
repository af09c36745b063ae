"""GPU (B200) parity AT THE BENCHMARKED CONFIGURATION: the reference's own random initialisation (torch.manual_seed(0) +
stock constructor — mdvit_b200.model.MDViT reproduces those weights bit for bit, tests/test_module_contract.py), 256x256,
train mode, against tests/golden/mdvit_randinit_golden.npz produced by the UNMODIFIED reference
(oracle/make_golden_randinit.py), and — at the bench's batch (32 images x 4 domains, stacked forward, CUDA-graph replay)
— against the fp32 oracle on the same GPU.

At this init the activations are not O(1): logits reach |x| ~ 200 (main) / ~ 90 (aux) and most sigmoids are saturated
(SURVEY.md section 0.8), so errors are normalised by the tensor abs-max, as BASELINE.json's north_star example
("max relative error <= 1e-2 on logits") must be read for such tensors.  The tolerances below are the measured margins
(DESIGN.md section 7) times ~2.
"""
import os

import numpy as np
import pytest
import torch

from mdvit_b200 import synth
from oracle.golden_sample import at_sample, rel_max
from tests.helpers import fingerprint

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

LOGIT_MAX_TOL = 1.0e-2       # max|out - ref| / max|ref| at 256x256, random init: north_star's example tolerance.  Measured: main
LOGIT_L2_TOL = 1.0e-2        # logits 1.8-3.0e-3 (L2 2.1-2.3e-3), aux logits 4.3-5.5e-3 (L2 4.0-4.6e-3)
TRAJ_LOSS_TOL = 5e-3         # per-step per-domain (L_seg, L_aux, L_kt) relative to the reference value; measured <= 1.5e-3
TRAJ_DICE_TOL = 1e-3         # Dice of the thresholded prediction after EVERY one of the 5 steps (north_star: "Dice within 1e-3");
                             # measured <= 6e-4
PARAM_FP_TOL = 5e-3          # per-parameter fingerprint (norm, probe projection) after 5 AdamW steps, weights
PARAM_FP_TOL_BIAS = 8e-2     # ... biases: zero-initialised, so after 5 steps the whole tensor IS 5 AdamW updates of +-lr-sized
                             # elements, and every element whose gradient sign sits inside the bf16 noise differs by 2*lr:
                             # measured worst 3.6e-2 (norm1.bias of stage 0); see zero_grad_param for the exactly-zero ones


def zero_grad_param(name):
    """Biases whose TRUE gradient is identically zero: a per-channel constant in front of a train-mode BatchNorm is removed
    by the mean subtraction (bridge.{0,3}.bias -> bridge.{1,4}; debranch*.linear{1-4}.bias and linear_fuse.0.bias -> the
    BatchNorm of linear_fuse).  Their computed gradient is round-off noise in the reference as well, and AdamW's
    g / sqrt(v) normalisation turns noise into +-lr steps: after 5 steps these tensors are 5e-4-sized noise on BOTH sides
    and cannot be compared element-wise.  They are checked to stay within AdamW's 5 * lr bound instead."""
    return name in ("bridge.0.bias", "bridge.3.bias") or (name.startswith("debranch") and name.endswith(".bias")
                                                            and (".linear_fuse.0." in name or name.split(".")[1] in ("linear1", "linear2", "linear3", "linear4")))


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return torch.device("cuda")


@pytest.fixture(scope="module")
def rgold():
    return np.load(os.path.join(ROOT, "tests", "golden", "mdvit_randinit_golden.npz"), allow_pickle=False)


def build_randinit(dev, seed=0, img=256):
    from mdvit_b200.model import MDViT
    torch.manual_seed(seed)
    m = MDViT(img_size=img, drop_rate=0.0, drop_path_rate=0.0, adapt_method="Sup", num_domains=4, decoder_name="MLPFM")
    for k in range(1, 5):
        getattr(m, f"debranch{k}").dropout.p = 0.0
    return m.to(dev).train()


def onehot(d, B, dev):
    return torch.nn.functional.one_hot(torch.full((B,), d), 4).float().to(dev)


def logits_errors(dev, rgold):
    m = build_randinit(dev)
    rows = []
    with torch.no_grad():
        for d in range(4):
            img, _ = synth.synth_batch(4321, d, 4, 256, 256)
            out, aux = m(img.to(dev), onehot(d, 4, dev), str(d))
            for name, t in (("out", out), ("aux", aux)):
                key = f"logits256_{name}_{d}"          # (the golden keeps a seeded sample of the elements)
                ts, ref = at_sample(t, rgold, key)
                rows.append((d, name, rel_max(t, rgold, key), ((ts - ref).norm() / ref.norm()).item(),
                             ((ts > 0) != (ref > 0)).float().mean().item()))
    return rows


def test_train_logits_256_random_init_vs_reference_golden(dev, rgold):
    """(i) train-mode logits, B=4, all four domains, reference random init."""
    rows = logits_errors(dev, rgold)
    for d, name, emax, el2, flips in rows:
        assert emax < LOGIT_MAX_TOL and el2 < LOGIT_L2_TOL, rows


def run_trajectory(dev, steps=5, **kw):
    from mdvit_b200 import ops
    from mdvit_b200.train_step import MKDTrainer
    m = build_randinit(dev)
    tr = MKDTrainer(m, lr=1e-4, weight_decay=0.05, **kw)
    losses, dice = [], []
    for step in range(steps):
        batches = [tuple(t.to(dev) for t in synth.synth_batch(1234 + step, d, 4, 256, 256)) + (d,) for d in range(4)]
        l = tr.step(batches)
        losses.append(l.double().cpu().numpy())
        dice.append([[ops.dice_jaccard(ops.seg_counts(o, b[1]))[0], ops.dice_jaccard(ops.seg_counts(a, b[1]))[0]]
                     for (o, a), b in zip(tr.last_logits, batches)])
    return m, tr, np.asarray(losses), np.asarray(dice)


def test_five_step_mkd_adamw_trajectory_vs_reference_golden(dev, rgold):
    """(ii) 5 optimizer steps of the MKD step + AdamW (multi_train_MDViT.py:121-213) from the reference's random init: the
    per-domain losses, the Dice of the thresholded predictions, EVERY parameter and the BatchNorm running statistics."""
    m, tr, losses, dice = run_trajectory(dev)
    ref_l, ref_d = rgold["traj_losses"], rgold["traj_dice"]
    assert np.abs(losses - ref_l).max() < TRAJ_LOSS_TOL * np.abs(ref_l).max(), (losses - ref_l)
    assert np.abs(losses / ref_l - 1).max() < 5 * TRAJ_LOSS_TOL, (losses / ref_l - 1)
    assert np.abs(dice - ref_d).max() < TRAJ_DICE_TOL, (dice - ref_d)
    names = [str(n) for n in rgold["param_names"]]
    named = dict(m.named_parameters())
    fp = fingerprint([(n, named[n]) for n in names])
    ref_fp = rgold["traj_param_fp"]
    err_norm = np.abs(fp[:, 0] - ref_fp[:, 0]) / np.maximum(ref_fp[:, 0], 1e-6)
    # probe projection error relative to the tensor norm (the projection itself can be ~0)
    err_probe = np.abs(fp[:, 1] - ref_fp[:, 1]) / np.maximum(ref_fp[:, 0] * np.sqrt([named[n].numel() for n in names]), 1e-6)
    live = np.asarray([not zero_grad_param(n) for n in names])
    err = np.maximum(err_norm, err_probe)
    worst = sorted(zip(err[live], np.asarray(names)[live]))[-5:]
    is_bias = np.asarray([n.endswith(".bias") for n in names])
    assert live.sum() >= 432 - 26 and err[live & is_bias].max() < PARAM_FP_TOL_BIAS and err[live & ~is_bias].max() < PARAM_FP_TOL, worst
    for n in np.asarray(names)[~live]:           # zero-gradient biases: initialised to 0, moved by at most 5 * lr * (1 + wd) each
        assert float(named[n].detach().abs().max()) <= 5 * 1e-4 * 1.01, n
    sd = m.state_dict()
    bn_names = [str(n) for n in rgold["traj_bn_names"]]
    bfp, ref_b = fingerprint([(k, sd[k]) for k in bn_names]), rgold["traj_bn_fp"]
    assert (np.abs(bfp[:, 0] - ref_b[:, 0]) / np.maximum(ref_b[:, 0], 1e-6)).max() < 2e-2
    assert int(sd["stem.0.bn.num_batches_tracked"]) == 20


def oracle_sd_from_model(m, requires_grad):
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    if requires_grad:
        for k, v in sd.items():
            if v.is_floating_point() and "running" not in k:
                v.requires_grad_(True)
    for k in list(sd):
        ck = synth.canonical_key(k)
        if ck != k:
            sd[k] = sd[ck]
    return sd


def graph_step_vs_oracle(dev, B=32):
    """The bench's step (B images x 4 domains stacked through the trunk, whole step replayed as one CUDA graph) against the
    fp32 oracle's autograd on the same GPU, from the reference's random init.  Returns (losses, ref_losses, grad report)."""
    from oracle import mdvit_oracle as O
    from mdvit_b200.train_step import MKDTrainer
    from tests.test_model_gpu import grad_report
    m = build_randinit(dev)
    tr = MKDTrainer(m, lr=1e-4, weight_decay=0.05)
    batches = [tuple(t.to(dev) for t in synth.synth_batch(777, d, B, 256, 256)) + (d,) for d in range(4)]
    tr.capture(batches, warmup=1)
    sd = oracle_sd_from_model(m, requires_grad=True)         # capture() restored the initial weights
    losses = tr.step_graph(None).double().cpu().numpy()
    torch.cuda.synchronize()
    grads = {n: p.grad.detach().clone() for n, p in m.named_parameters()}
    # oracle, one domain graph at a time (gradients are additive over domains; DA parameters get only the 0.5 kt + 0.5 seg part)
    names = [k for k, v in sd.items() if v.requires_grad and synth.canonical_key(k) == k]
    ref_g = {n: torch.zeros_like(sd[n]) for n in names}
    ref_l = []
    for img, lab, d in batches:
        out, aux = O.mdvit_forward(sd, img, onehot(d, B, dev), str(d), training=True)
        ls, la, lk = O.seg_losses(out, aux, lab)
        ref_l.append([ls.item(), la.item(), lk.item()])
        g_aux = torch.autograd.grad(la, [sd[n] for n in names], retain_graph=True, allow_unused=True)
        g_uni = torch.autograd.grad(0.5 * lk + 0.5 * ls, [sd[n] for n in names], allow_unused=True)
        for n, ga, gu in zip(names, g_aux, g_uni):
            if gu is not None:
                ref_g[n] += gu
            if ga is not None and not O.is_da(n):
                ref_g[n] += ga
        del out, aux, ls, la, lk, g_aux, g_uni
    return losses, np.asarray(ref_l), grad_report(grads, ref_g)


def test_bench_config_graph_step_vs_fp32_oracle(dev):
    """(iii) B=32 x 4 domains, stacked forward, CUDA-graph replay with the WeightMirror — the configuration bench.py times
    (dropout off: its RNG stream cannot be matched) — losses and all gradients against the fp32 oracle on this GPU."""
    losses, ref_l, (g_all, w_tight, w_loose, text) = graph_step_vs_oracle(dev, B=32)
    assert np.abs(losses / ref_l - 1).max() < TRAJ_LOSS_TOL, (losses, ref_l)
    assert g_all < 0.05 and w_tight < 0.15 and w_loose < 0.15, (g_all, w_tight, w_loose, text)
