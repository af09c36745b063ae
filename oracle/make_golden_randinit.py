"""TEST INFRASTRUCTURE ONLY.  Generates tests/golden/mdvit_randinit_golden.npz by running the UNMODIFIED reference
(imported from /root/reference through oracle/ref_shim.py) in the build container, at the configuration bench.py
measures: the reference's OWN random initialisation (torch.manual_seed(0) + the stock constructor,
Models/Transformer/mdvit.py:484-504,648-664), 256x256 inputs, train mode (BatchNorm batch statistics).

    python oracle/make_golden_randinit.py

Contents
  init_fp                     [432,2] fingerprint (l2 norm, probe dot) of every parameter right after the constructor —
                              mdvit_b200.model.MDViT must reproduce the SAME weights from the same seed (bit-identical init)
  logits256_{out,aux}_{d}     train-mode logits [4,1,256,256] per domain d (fp16 storage: 5e-4 relative, tolerance is 1e-2)
  traj_losses                 [5,4,3] per step, per domain (L_seg, L_aux, L_kt)   (multi_train_MDViT.py:147-169)
  traj_dice                   [5,4,2] per step, per domain Dice of the thresholded main / aux prediction vs the label
                              (medpy.metric.binary.dc semantics, multi_train_MDViT.py:172-177)
  traj_param_fp               [432,2] parameter fingerprints after the 5 AdamW steps (multi_train_MDViT.py:93-94,213)
  traj_bn_fp                  BN running statistics fingerprints after the 5 steps (20 train forwards)
Dropout / DropPath / Dropout2d are disabled (torch RNG streams cannot be reproduced by another implementation).
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mdvit_b200 import synth  # noqa: E402
from oracle import ref_shim  # noqa: E402
from oracle.golden_sample import keep_samples  # noqa: E402
from oracle.make_golden import fingerprint  # noqa: E402

SEED, IMG, B, STEPS = 0, 256, 4, 5


# train-mode logits kept as a seeded sample of 1/8 of their elements (oracle/golden_sample.py)
SAMPLED = {f"logits256_{k}_{d}": 32768 for k in ("out", "aux") for d in range(4)}


def hard_dice(logits, label):
    """medpy.metric.binary.dc of (sigmoid(logits) > 0.5) vs label over the whole batch tensor."""
    pred = (torch.sigmoid(logits) > 0.5)
    lab = label > 0.5
    inter = (pred & lab).sum().item()
    den = pred.sum().item() + lab.sum().item()
    return 2.0 * inter / den if den > 0 else 0.0


def build(ref):
    torch.manual_seed(SEED)
    m = ref.MDViT(img_size=IMG, drop_rate=0.0, drop_path_rate=0.0, adapt_method="Sup", num_domains=4, decoder_name="MLPFM")
    for k in range(1, 5):
        getattr(m, f"debranch{k}").dropout.p = 0.0
    return m


def main():
    torch.set_num_threads(8)
    ref = ref_shim.load_reference()
    out = {}
    m = build(ref).train()
    named = list(m.named_parameters())
    out["param_names"] = np.asarray([n for n, _ in named])
    out["init_fp"] = fingerprint(named)
    # ---- (i) train-mode logits, 256x256, B=4, all four domains (BN running stats get updated: rebuild afterwards)
    with torch.no_grad():
        for d in range(4):
            img, _ = synth.synth_batch(4321, d, B, IMG, IMG)
            dl = torch.nn.functional.one_hot(torch.full((B,), d), 4).float()
            o, a = m(img, dl, str(d))
            out[f"logits256_out_{d}"], out[f"logits256_aux_{d}"] = o.numpy().astype(np.float16), a.numpy().astype(np.float16)
            out[f"logits256_absmax_{d}"] = np.asarray([o.abs().max().item(), a.abs().max().item()])
            print("logits", d, out[f"logits256_absmax_{d}"], flush=True)
    # ---- (ii) 5-step MKD + AdamW trajectory (multi_train_MDViT.py:121-213)
    m = build(ref).train()
    opt = torch.optim.AdamW(m.parameters(), lr=1e-4, weight_decay=0.05)
    losses, dice = [], []
    for step in range(STEPS):
        batches = [synth.synth_batch(1234 + step, d, B, IMG, IMG) + (d,) for d in range(4)]
        opt.zero_grad()
        # reference_step restates multi_train_MDViT.py:129-207 around the unmodified model; hook the logits for Dice
        logits = []
        h = m.register_forward_hook(lambda mod, inp, o: logits.append((o[0].detach(), o[1].detach())))
        L = ref_shim.reference_step(m, batches, ref.dice_loss)
        h.remove()
        opt.step()
        losses.append([[s.item(), a.item(), k.item()] for s, a, k in zip(L["seg_each"], L["aux_each"], L["kt_each"])])
        dice.append([[hard_dice(o, b[1]), hard_dice(a, b[1])] for (o, a), b in zip(logits, batches)])
        print("step", step, np.asarray(losses[-1]).round(4).tolist(), np.asarray(dice[-1]).round(4).tolist(), flush=True)
    out["traj_losses"] = np.asarray(losses, np.float64)
    out["traj_dice"] = np.asarray(dice, np.float64)
    out["traj_param_fp"] = fingerprint(list(m.named_parameters()))
    sd = m.state_dict()
    bn_keys = [k for k in sd if k.endswith("running_mean") or k.endswith("running_var")]
    out["traj_bn_names"] = np.asarray(bn_keys)
    out["traj_bn_fp"] = fingerprint([(k, sd[k]) for k in bn_keys])
    keep_samples(out, SAMPLED)
    path = os.path.join(ROOT, "tests", "golden", "mdvit_randinit_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB;", len(out), "arrays")


if __name__ == "__main__":
    main()
