"""TEST INFRASTRUCTURE ONLY.  Golden logits of the UNMODIFIED reference MDViT_DSN (domain-specific norms,
Models/Transformer/mdvit.py:735-960) -> tests/golden/mdvit_dsn_golden.npz.   python oracle/make_golden_dsn.py

Weights: torch.manual_seed(0) + the stock constructor (mdvit_b200.model.MDViT_DSN reproduces them bit for bit), then
synth.dsn_perturb so that the four norm sets differ.  Dropout2d of the aux decoders off."""
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

# the 256x256 DeepLabV3 logits kept as a seeded sample of 1/8 of their elements (oracle/golden_sample.py)
SAMPLED = {"dl_eval_out": 16384, "dl_eval_aux": 16384, "dl_train_aux": 16384}


def aux_state(model, prefix="debranch"):
    """Deterministic weights for the auxiliary-decoder tensors of a model (synth_tensor handles any key/shape)."""
    return {k: synth.synth_tensor(k, tuple(v.shape)) for k, v in model.state_dict().items() if k.startswith(prefix)}


def mlp_aux_state(model):
    return aux_state(model, "debranch")


def main():
    ref_shim.load_reference()
    from Models.Transformer.mdvit import MDViT_DSN
    torch.manual_seed(0)
    m = MDViT_DSN(img_size=64, adapt_method="Sup", num_domains=4, decoder_name="MLPFM")
    out = {"keys": np.asarray(list(m.state_dict().keys())), "init_fp": fingerprint(list(m.named_parameters()))}
    m.load_state_dict(synth.dsn_perturb(m.state_dict()), strict=True)
    for k in range(1, 5):
        getattr(m, f"debranch{k}").dropout.p = 0.0
    with torch.no_grad():
        for mode in ("eval", "train"):
            m.train(mode == "train")
            for d in (1, 3):
                img, _ = synth.synth_batch(11, d, 2, 64, 64)
                dl = torch.nn.functional.one_hot(torch.full((2,), d), 4).float()
                o, a = m(img, dl, str(d))
                out[f"{mode}_out_{d}"], out[f"{mode}_aux_{d}"] = o.numpy(), a.numpy()
    # ---- MDViT with the 'MLP' auxiliary decoder (Decoders.MLPDecoder, Decoders.py:239-286; mdvit.py:607-611)
    from Models.Transformer.mdvit import MDViT
    m = MDViT(img_size=64, adapt_method="Sup", num_domains=4, decoder_name="MLP")
    m.load_state_dict(synth.synth_state_dict(0, aux=False) | {k: v for k, v in mlp_aux_state(m).items()}, strict=True)
    for k in range(1, 5):
        getattr(m, f"debranch{k}").dropout.p = 0.0
    out["mlp_keys"] = np.asarray(list(m.state_dict().keys()))
    with torch.no_grad():
        for mode in ("eval", "train"):
            m.train(mode == "train")
            img, _ = synth.synth_batch(12, 2, 2, 64, 64)
            dl = torch.nn.functional.one_hot(torch.full((2,), 2), 4).float()
            o, a = m(img, dl, "2")
            out[f"mlp_{mode}_out"], out[f"mlp_{mode}_aux"] = o.numpy(), a.numpy()
    # ---- MDViT with the 'Transformer' auxiliary decoder (mdvit.py:613-642,704-712): one extra 4-stage decoder per domain
    torch.manual_seed(0)
    m = MDViT(img_size=64, adapt_method="Sup", num_domains=4, decoder_name="Transformer")
    out["tr_keys"] = np.asarray(list(m.state_dict().keys()))
    out["tr_init_fp"] = fingerprint(list(m.named_parameters()))
    m.load_state_dict(synth.synth_state_dict(0, aux=False) | aux_state(m, "debranchs"), strict=True)
    with torch.no_grad():
        for mode in ("eval", "train"):
            m.train(mode == "train")
            for d in (0, 3):
                img, _ = synth.synth_batch(14, d, 2, 64, 64)
                dl = torch.nn.functional.one_hot(torch.full((2,), d), 4).float()
                o, a = m(img, dl, str(d))
                out[f"tr_{mode}_out_{d}"], out[f"tr_{mode}_aux_{d}"] = o.numpy(), a.numpy()
    # ---- MDViT with the 'DeepLabV3' auxiliary decoder (mdvit.py:608-611, Decoders.py:218-235, Utils/_deeplab.py:115-166).  256x256 so
    # that the last encoder map is 8x8 and the dilation-6 taps land inside it; ASPP's Dropout(0.1) off.  Besides the logits: the
    # gradients of sum(aux * R) w.r.t. every parameter of the active branch and w.r.t. the stem (through the whole encoder).
    torch.manual_seed(0)
    m = MDViT(img_size=256, adapt_method="Sup", num_domains=4, decoder_name="DeepLabV3")
    out["dl_keys"] = np.asarray(list(m.state_dict().keys()))
    out["dl_init_fp"] = fingerprint(list(m.named_parameters()))
    m.load_state_dict(synth.synth_state_dict(0, aux=False) | aux_state(m, "debranch"), strict=True)
    for k in range(1, 5):
        getattr(m, f"debranch{k}").classifier[0].project[3].p = 0.0
    img, _ = synth.synth_batch(15, 1, 2, 256, 256)
    dl = torch.nn.functional.one_hot(torch.full((2,), 1), 4).float()
    with torch.no_grad():
        m.eval()
        o, a = m(img, dl, "1")
        out["dl_eval_out"], out["dl_eval_aux"] = o.numpy().astype(np.float16), a.numpy().astype(np.float16)
        out["dl_eval_absmax"] = np.asarray([o.abs().max().item(), a.abs().max().item()])
    m.train()
    o, a = m(img, dl, "1")
    out["dl_train_aux"] = a.detach().numpy().astype(np.float16)
    out["dl_train_absmax"] = np.asarray([a.abs().max().item()])
    R = synth.synth_tensor("dl_probe", tuple(a.shape))
    (a * R).sum().backward()
    gnames = [n for n, p in m.named_parameters() if n.startswith("debranch2.") or n.startswith("stem.")]
    out["dl_grad_names"] = np.asarray(gnames)
    out["dl_grad_fp"] = fingerprint([(n, dict(m.named_parameters())[n].grad) for n in gnames])
    # ---- BASE_DSN (Models/Transformer/base.py:515-696): the DSN trunk without auxiliary branches, Sup and plain attention
    from Models.Transformer.base import BASE_DSN
    for am in ("Sup", None):
        tag = "sup" if am else "plain"
        torch.manual_seed(0)
        m = BASE_DSN(img_size=64, adapt_method=am, num_domains=4)
        out[f"base_dsn_{tag}_keys"] = np.asarray(list(m.state_dict().keys()))
        out[f"base_dsn_{tag}_init_fp"] = fingerprint(list(m.named_parameters()))
        m.load_state_dict(synth.dsn_perturb(m.state_dict()), strict=True)
        with torch.no_grad():
            for mode in ("eval", "train"):
                m.train(mode == "train")
                for d in (0, 2):
                    img, _ = synth.synth_batch(13, d, 2, 64, 64)
                    dl = torch.nn.functional.one_hot(torch.full((2,), d), 4).float() if am else None
                    out[f"base_dsn_{tag}_{mode}_{d}"] = m(img, dl, str(d)).numpy()
    keep_samples(out, SAMPLED)
    path = os.path.join(ROOT, "tests", "golden", "mdvit_dsn_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
