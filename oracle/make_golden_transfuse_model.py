"""TEST INFRASTRUCTURE ONLY.  Golden vectors for the whole TransFuse_S_adapt (Models/Hybrid_models/TransFuseFolder/TransFuse.py:
182-283) and structure_loss (multi_train_TransFuse.py:29-38): runs the UNMODIFIED reference from /root/reference in the build
container at ITS OWN random init (torch.manual_seed(0), stock constructor, drop_rate=0 so that the forward is deterministic)
and writes tests/golden/transfuse_model_golden.npz and tests/golden/transfuse_structure_loss_golden.npz.

    python oracle/make_golden_transfuse_model.py

The tests rebuild the same weights by constructing mdvit_b200.transfuse.TransFuse_S_adapt under the same seed (the init
fingerprints in the file prove the two constructors draw identical weights) and the same inputs from the numpy streams below."""
import os
import sys
import zlib

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _t(key, shape, std=1.0):
    g = np.random.Generator(np.random.PCG64([2025, zlib.crc32(key.encode())]))
    return torch.from_numpy((g.standard_normal(shape) * std).astype(np.float32))


def case(B=2, side=256):
    """image, binary mask (a disc per sample, so that the 31x31 box filter sees edges) and one-hot domain labels"""
    img = _t("tfm_img", (B, 3, side, side))
    yy, xx = torch.meshgrid(torch.arange(side), torch.arange(side), indexing="ij")
    mask = torch.stack([(((yy - side * (0.4 + 0.1 * b)) ** 2 + (xx - side * (0.55 - 0.1 * b)) ** 2) < (side * (0.22 + 0.06 * b)) ** 2).float()
                        for b in range(B)]).unsqueeze(1)
    dom = torch.tensor([(1 + 2 * b) % 4 for b in range(B)])
    return img, mask, F.one_hot(dom, 4).float()


def structure_loss_ref(pred, mask):
    """verbatim semantics of multi_train_TransFuse.py:29-38 (the trainer file itself cannot be imported: its dataset import is broken
    upstream, SURVEY.md section 8(f)); checked against it textually"""
    weit = 1 + 5 * torch.abs(F.avg_pool2d(mask, kernel_size=31, stride=1, padding=15) - mask)
    wbce = F.binary_cross_entropy_with_logits(pred, mask, reduction='none')
    wbce = (weit * wbce).sum(dim=(2, 3)) / weit.sum(dim=(2, 3))
    pred = torch.sigmoid(pred)
    inter = ((pred * mask) * weit).sum(dim=(2, 3))
    union = ((pred + mask) * weit).sum(dim=(2, 3))
    wiou = 1 - (inter + 1) / (union - inter + 1)
    return (wbce + wiou).mean()


def structure_loss_golden(maps, mask):
    """structure_loss_ref and its gradient, with the 0.5/0.3/0.2 weights of multi_train_TransFuse.py:169-172, on the reference's
    maps rounded to fp16: the loss reads every pixel, so its input is stored whole, and in fp16 to keep the file small."""
    from oracle.golden_sample import keep_samples
    preds = [torch.from_numpy(np.asarray(p, np.float16).astype(np.float32)).requires_grad_(True) for p in maps]
    losses = [structure_loss_ref(p, mask) for p in preds]
    loss = 0.5 * losses[2] + 0.3 * losses[1] + 0.2 * losses[0]
    loss.backward()
    out = {"losses": np.asarray([l.item() for l in losses] + [loss.item()], np.float64)}
    for n, p in zip(("x", "1", "2"), preds):
        out["pred_" + n] = p.detach().numpy().astype(np.float16)
        out["dpred_" + n] = p.grad.numpy().astype(np.float32)
    keep_samples(out, {"dpred_" + n: 16384 for n in ("x", "1", "2")})
    return out


KEEP_FULL = ("resnet.conv1.weight", "resnet.bn1.weight", "resnet.layer1.0.conv1.weight", "resnet.layer2.0.downsample.0.weight",
             "resnet.layer3.5.bn2.bias", "up1.conv.identity.0.weight", "up_c.fc1.weight", "up_c.fc2.bias", "up_c.spatial.conv.weight",
             "up_c.spatial.bn.weight", "up_c.W_g.conv.bias", "up_c.residual.bn1.weight", "up_c.residual.conv3.conv.weight",
             "up_c_1_2.attn_block.psi.0.weight", "up_c_1_2.attn_block.psi.1.weight", "up_c_2_2.attn_block.W_x.0.weight",
             "final_x.2.conv.weight", "final_1.1.conv.bias", "final_2.0.bn.weight", "transformer.norm.weight",
             "transformer.blocks.0.attn.domain_layer.2.bias", "transformer.patch_embed.proj.bias")
# the maps and the larger of the gradients above kept as seeded samples of their elements (oracle/golden_sample.py)
SAMPLED = {**{n: 16384 for n in ("map_x", "map_1", "map_2", "eval_map_x", "eval_map_1", "eval_map_2")},
           **{"grad." + n: 8192 for n in ("resnet.conv1.weight", "resnet.layer1.0.conv1.weight", "up1.conv.identity.0.weight",
                                          "up_c.fc1.weight", "up_c.residual.conv3.conv.weight")}}


def save(out, mask):
    """Writes both golden files from the reference's outputs (`out` holds full tensors; it is sampled in place)."""
    from oracle.golden_sample import keep_samples
    sl = structure_loss_golden([out[n] for n in ("map_x", "map_1", "map_2")], mask)
    keep_samples(out, SAMPLED)
    for name, d in (("transfuse_model_golden.npz", out), ("transfuse_structure_loss_golden.npz", sl)):
        path = os.path.join(ROOT, "tests", "golden", name)
        np.savez_compressed(path, **d)
        print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def main():
    from oracle import ref_shim
    from oracle.make_golden import fingerprint
    ref_shim.install_stubs()
    sys.dont_write_bytecode = True
    sys.path.insert(0, ref_shim.REFERENCE_ROOT)
    from Models.Hybrid_models.TransFuseFolder.TransFuse import TransFuse_S_adapt
    torch.manual_seed(0)
    m = TransFuse_S_adapt(drop_rate=0.0, pretrained=False, num_domains=4).train()
    out = {"keys": np.asarray(list(m.state_dict().keys())),
           "init_fp": fingerprint(list(m.named_parameters()))}
    img, mask, dlab = case()
    maps = m(img, dlab)
    losses = [structure_loss_ref(p, mask) for p in maps]
    loss = 0.5 * losses[2] + 0.3 * losses[1] + 0.2 * losses[0]      # multi_train_TransFuse.py:169-172 (maps are (4, 3, 2))
    for n, p in zip(("map_x", "map_1", "map_2"), maps):
        out[n] = p.detach().numpy().astype(np.float32)
    out["losses"] = np.asarray([l.item() for l in losses] + [loss.item()], np.float64)
    loss.backward()
    named = [(n, p.grad) for n, p in m.named_parameters() if p.grad is not None]
    out["grad_names"] = np.asarray([n for n, _ in named])
    out["grad_fp"] = fingerprint(named)
    for n, g in named:
        if n in KEEP_FULL:
            out["grad." + n] = g.numpy().astype(np.float32)
    sd = m.state_dict()
    for k in ("resnet.bn1.running_mean", "resnet.bn1.running_var", "resnet.layer3.5.bn2.running_var", "up_c.spatial.bn.running_mean",
              "up_c.residual.bn1.running_var", "up_c_1_2.attn_block.psi.1.running_var", "final_x.0.bn.running_mean"):
        out["buf." + k] = sd[k].numpy().astype(np.float32)
    # eval-mode maps (running statistics after the one training forward above)
    m.eval()
    with torch.no_grad():
        emaps = m(img, dlab)
    for n, p in zip(("eval_map_x", "eval_map_1", "eval_map_2"), emaps):
        out[n] = p.numpy().astype(np.float16)
    out["eval_absmax"] = np.asarray([p.abs().max().item() for p in emaps])
    print("losses", out["losses"], "map absmax", [float(np.abs(out[n]).max()) for n in ("map_x", "map_1", "map_2")])
    save(out, mask)


if __name__ == "__main__":
    main()
