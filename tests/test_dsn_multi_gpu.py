"""MDViT_DSN / BASE_DSN stacked multi-domain pass: the per-group LayerNorm / BatchNorm kernels (one parameter set per row
group, mdv_*_gp) against torch fp32 slice by slice, forward_multi against G separate forwards, and the fused MKDTrainer step
against the per-domain loop.  The models are loaded with synth.dsn_perturb: with identical norm sets a kernel reading the
wrong set would be invisible."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from mdvit_b200 import synth
from tests.test_model_gpu import grad_report, rel, rel_l2

F32_TOL = 2e-4
BF16_TOL = 1e-2


@pytest.fixture(scope="module")
def env():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    from mdvit_b200 import _lib as L
    return L, L.lib(), torch.device("cuda")


def _fake_table(addrs):
    from mdvit_b200 import _lib as L
    t = L.PtrTable()
    for i, a in enumerate(addrs):
        t.p[i] = a
    return t


def test_gp_entry_points_reject_bad_group_counts_and_missing_parameters(built_lib):
    """Argument validation happens before any CUDA call: G outside 1..8 and a missing gamma / beta of a used group return
    MDV_ERR_ARG (-1).  The pointers are never dereferenced."""
    lib = built_lib
    p = [ctypes.c_void_p(0x10000 * (i + 1)) for i in range(8)]
    sets = _fake_table([0x100000 + 0x1000 * g for g in range(8)])
    sets2 = _fake_table([0x200000 + 0x1000 * g for g in range(8)])
    for G in (0, 9):
        assert lib.mdv_layernorm_fwd_gp(p[0], sets, sets2, 1e-6, p[1], p[2], p[3], G, 64, 64, None) == -1
        assert lib.mdv_layernorm_bwd_gp(p[0], p[1], p[2], p[3], sets, None, p[4], None, None, 1, 0.0, None, 0, sets2, _fake_table([]), None,
                                        G, 64, 64, None) == -1
        assert lib.mdv_bn_train_fwd_gp(p[0], G, 64, 64, 1e-5, 0.1, _fake_table([]), _fake_table([]), _fake_table([]), sets, sets2, 3, p[1],
                                       p[2], p[3], 0, p[4], None) == -1
        assert lib.mdv_bn_act_bwd_gp(p[0], p[1], p[2], p[3], sets, sets2, 3, p[4], 0, _fake_table([]), _fake_table([]), G, 64, 64, p[5],
                                     None) == -1
    # a missing gamma / beta of a used group
    assert lib.mdv_layernorm_fwd_gp(p[0], _fake_table([0x500000]), sets2, 1e-6, p[1], p[2], p[3], 2, 64, 64, None) == -1
    assert lib.mdv_bn_train_fwd_gp(p[0], 2, 64, 64, 1e-5, 0.1, _fake_table([]), _fake_table([]), _fake_table([]), sets, _fake_table([0x500000]),
                                   3, p[1], p[2], p[3], 0, p[4], None) == -1
    assert lib.mdv_bn_act_bwd_gp(p[0], p[1], p[2], p[3], _fake_table([0x500000]), sets2, 3, p[4], 0, _fake_table([]), _fake_table([]), 2, 64, 64,
                                 p[5], None) == -1


# ------------------------------------------------------------------------------------------------- kernels
@pytest.mark.gpu
@pytest.mark.parametrize("Mg,C", [(37, 64), (37, 128), (37, 320), (37, 512), (1003, 320), (32 * 4096, 64)])
def test_layernorm_gp_matches_torch_per_slice(env, Mg, C):
    """G = 4 row groups, group g normalised with (gamma[g], beta[g]); dgamma[g] / dbeta[g] accumulate into pre-filled buffers
    and NULL targets are skipped; the shared bias gradient (dbias_masked) is one sum over all rows.  Mg = 37 is not a multiple
    of any rows-per-block of the kernels, so row chunks would straddle group boundaries if the grid allowed it."""
    L, lib, dev = env
    G, M = 4, 4 * Mg
    torch.manual_seed(Mg + C)
    x = (torch.randn(M, C, device=dev) * 2 + 0.5).requires_grad_()
    gs = [(1 + 0.3 * torch.randn(C, device=dev)).requires_grad_() for _ in range(G)]
    bs = [(0.3 * torch.randn(C, device=dev)).requires_grad_() for _ in range(G)]
    y = torch.empty(M, C, device=dev, dtype=torch.bfloat16)
    mean, rstd = torch.empty(M, device=dev), torch.empty(M, device=dev)
    L.check(lib.mdv_layernorm_fwd_gp(L.ptr(x), L.ptr_table(gs), L.ptr_table(bs), 1e-6, L.ptr(y), L.ptr(mean), L.ptr(rstd), G, Mg, C,
                                     L.stream()), "ln_gp")
    ref = torch.cat([F.layer_norm(x[g * Mg:(g + 1) * Mg], (C,), gs[g], bs[g], 1e-6) for g in range(G)])
    for g in range(G):
        assert rel(y[g * Mg:(g + 1) * Mg], ref[g * Mg:(g + 1) * Mg]) < BF16_TOL, g
    dy, dres = torch.randn(M, C, device=dev), torch.randn(M, C, device=dev)
    (ref * dy).sum().backward()
    pre_g = [torch.randn(C, device=dev) for _ in range(G)]
    pre_b = [torch.randn(C, device=dev) for _ in range(G)]
    dgs, dbs = [t.clone() for t in pre_g], [t.clone() for t in pre_b]
    dg_t, db_t = list(dgs), list(dbs)
    dg_t[1], db_t[2] = None, None          # frozen / da_only targets: not written
    dx, dxm = torch.empty(M, C, device=dev), torch.empty(M, C, device=dev, dtype=torch.bfloat16)
    dbm = torch.ones(C, device=dev)
    L.check(lib.mdv_layernorm_bwd_gp(L.ptr(dy), L.ptr(x), L.ptr(mean), L.ptr(rstd), L.ptr_table(gs), L.ptr(dres), L.ptr(dx), L.ptr(dxm), None,
                                     1, 0.0, None, 0, L.ptr_table(dg_t), L.ptr_table(db_t), L.ptr(dbm), G, Mg, C, L.stream()), "ln_bwd_gp")
    want_dx = x.grad + dres
    for g in range(G):
        s = slice(g * Mg, (g + 1) * Mg)
        assert rel(dx[s], want_dx[s]) < F32_TOL, g
        assert rel(dgs[g], pre_g[g] + (gs[g].grad if g != 1 else 0)) < F32_TOL, g
        assert rel(dbs[g], pre_b[g] + (bs[g].grad if g != 2 else 0)) < F32_TOL, g
    assert rel(dxm, want_dx) < BF16_TOL
    assert rel(dbm, 1 + want_dx.sum(0)) < 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("Mg,C,act,bf16", [(512, 32, 3, False), (1000, 64, 3, True), (77, 128, 3, False), (3000, 320, 2, False),
                                           (2048, 512, 2, True)])
def test_batchnorm_gp_matches_batchnorm2d_per_slice(env, Mg, C, act, bf16):
    """Group g of [4*Mg, C] against its own nn.BatchNorm2d (train mode): outputs, dz, dgamma / dbeta (accumulated into pre-filled
    buffers, NULL entries skipped), and each group's running buffers and num_batches_tracked — no group touches another's.
    `bf16` selects bf16 y and dz instead of fp32 (the model's backward writes dz in bf16)."""
    L, lib, dev = env
    G, M = 4, 4 * Mg
    torch.manual_seed(Mg + C)
    z = (torch.randn(M, C, device=dev) * 2 + 0.5).requires_grad_()
    bns = [torch.nn.BatchNorm2d(C).to(dev).train() for _ in range(G)]
    with torch.no_grad():
        for k, bn in enumerate(bns):
            bn.weight.copy_(1 + 0.3 * torch.randn(C, device=dev))
            bn.bias.copy_(0.3 * torch.randn(C, device=dev))
            bn.running_mean.copy_(0.2 * torch.randn(C, device=dev))
            bn.running_var.copy_(1 + 0.3 * torch.rand(C, device=dev))
            bn.num_batches_tracked.fill_(3 * k)
    rm = [bn.running_mean.clone() for bn in bns]
    rv = [bn.running_var.clone() for bn in bns]
    nbt = [bn.num_batches_tracked.clone() for bn in bns]
    gam = [bn.weight.detach().clone() for bn in bns]
    bet = [bn.bias.detach().clone() for bn in bns]
    mean, rstd = torch.empty(G, C, device=dev), torch.empty(G, C, device=dev)
    y = torch.empty(M, C, device=dev, dtype=torch.bfloat16 if bf16 else torch.float32)
    ws = torch.empty(3 * C * G, dtype=torch.float64, device=dev)
    L.check(lib.mdv_bn_train_fwd_gp(L.ptr(z), G, Mg, C, 1e-5, 0.1, L.ptr_table(rm), L.ptr_table(rv), L.ptr_table(nbt), L.ptr_table(gam),
                                    L.ptr_table(bet), act, L.ptr(mean), L.ptr(rstd), L.ptr(y), int(bf16), L.ptr(ws), L.stream()), "bn_gp")
    actf = F.relu if act == 2 else F.hardswish
    ref = torch.cat([actf(bns[g](z[g * Mg:(g + 1) * Mg].view(Mg, C, 1, 1))).view(Mg, C) for g in range(G)])
    for g in range(G):
        s = slice(g * Mg, (g + 1) * Mg)
        assert rel(y[s], ref[s]) < (BF16_TOL if bf16 else F32_TOL), g
        assert rel(rm[g], bns[g].running_mean) < 1e-5 and rel(rv[g], bns[g].running_var) < 1e-5, g
        assert int(nbt[g]) == int(bns[g].num_batches_tracked) == 3 * g + 1, g
    dy = torch.randn(M, C, device=dev)
    (ref * dy).sum().backward()
    pre = [torch.randn(C, device=dev) for _ in range(2 * G)]
    dgs, dbs = [t.clone() for t in pre[:G]], [t.clone() for t in pre[G:]]
    dz = torch.empty(M, C, device=dev, dtype=torch.bfloat16 if bf16 else torch.float32)
    L.check(lib.mdv_bn_act_bwd_gp(L.ptr(dy), L.ptr(z), L.ptr(mean), L.ptr(rstd), L.ptr_table(gam), L.ptr_table(bet), act, L.ptr(dz), int(bf16),
                                  L.ptr_table([dgs[0], None, dgs[2], dgs[3]]), L.ptr_table([None, dbs[1], dbs[2], None]), G, Mg, C, L.ptr(ws),
                                  L.stream()), "bn_bwd_gp")
    for g in range(G):
        s = slice(g * Mg, (g + 1) * Mg)
        assert rel(dz[s], z.grad[s]) < (BF16_TOL if bf16 else 1e-3), g
        assert rel(dgs[g], pre[g] + (bns[g].weight.grad if g != 1 else 0)) < 1e-3, g
        want_b = pre[G + g] + (bns[g].bias.grad if g in (1, 2) else 0)
        assert rel(dbs[g], want_b) < 1e-3, g


# ------------------------------------------------------------------------------------------------- models
def _dsn(dev, kind, am="Sup"):
    from mdvit_b200.model import BASE_DSN, MDViT_DSN
    torch.manual_seed(0)
    m = MDViT_DSN(img_size=64, adapt_method=am, num_domains=4, decoder_name="MLPFM") if kind == "mdvit" else \
        BASE_DSN(img_size=64, adapt_method=am, num_domains=4)
    m.load_state_dict(synth.dsn_perturb(m.state_dict()), strict=True)
    for k in range(1, 5):
        if hasattr(m, f"debranch{k}"):
            getattr(m, f"debranch{k}").dropout.p = 0.0
    return m.to(dev)


def _onehot(d, B, dev):
    return F.one_hot(torch.full((B,), d), 4).float().to(dev)


CASES = [("mdvit", "Sup"), ("base", "Sup"), ("base", None)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,am", CASES)
def test_dsn_forward_multi_equals_per_domain_forwards(env, kind, am):
    """Train mode: one stacked pass (row group g uses norm set int(domains[g])) against 4 separate forwards on an identical copy:
    logits, aux logits, every running buffer of every norm set, and num_batches_tracked == 1 per set.  Eval mode: forward_multi
    returns the separate forwards."""
    _, _, dev = env
    m1, m2 = _dsn(dev, kind, am).train(), _dsn(dev, kind, am).train()
    doms = [2, 0, 3, 1]          # not in set order: group g must read set int(domains[g]), not set g
    batches = [tuple(t.to(dev) for t in synth.synth_batch(1, d, 2, 64, 64)) + (d,) for d in doms]
    x = torch.cat([b[0] for b in batches])
    dl = torch.cat([_onehot(d, 2, dev) for d in doms]) if am else None

    def sep_forward(m):
        res = []
        for img, _, d in batches:
            o = m(img, _onehot(d, 2, dev) if am else None, str(d))
            res.append(tuple(o) if isinstance(o, list) else (o, None))
        return res

    with torch.no_grad():
        sep = sep_forward(m1)
        fused = m2.forward_multi(x, dl, [str(d) for d in doms])
    assert len(fused) == 4
    for (o1, a1), (o2, a2) in zip(sep, fused):
        assert o2.shape == o1.shape and rel_l2(o2, o1) < 5e-3
        if kind == "mdvit":
            assert rel_l2(a2, a1) < 1e-2
        else:
            assert a1 is None and a2 is None
    sd1, sd2 = m1.state_dict(), m2.state_dict()
    n_sets = 0
    for k in sd1:
        if "running" in k:
            assert rel(sd2[k], sd1[k]) < 5e-3, k
        if k.endswith("num_batches_tracked"):
            assert int(sd1[k]) == int(sd2[k]) == 1, k
            n_sets += 1
    assert n_sets >= 4 * 12          # stem 2, patch embeddings 4, bridge 2, decoder convs 4 BatchNorms per set
    m2.load_state_dict(m1.state_dict())
    m1.eval(), m2.eval()
    with torch.no_grad():
        sep = sep_forward(m1)
        fused = m2.forward_multi(x, dl, [str(d) for d in doms])
    for (o1, a1), (o2, a2) in zip(sep, fused):
        assert rel(o2, o1) < 1e-5 and (a1 is None or rel(a2, a1) < 1e-5)


@pytest.mark.gpu
def test_dsn_forward_multi_rejects_repeated_domains(env):
    _, _, dev = env
    m = _dsn(dev, "base").train()
    x = torch.cat([synth.synth_batch(1, d, 2, 64, 64)[0] for d in (0, 1, 0)]).to(dev)
    dl = torch.cat([_onehot(d, 2, dev) for d in (0, 1, 0)])
    with pytest.raises(ValueError):
        m.forward_multi(x, dl, ["0", "1", "0"])
    with pytest.raises(ValueError):
        m.eval().forward_multi(x, dl, ["0", "1", "0"])


# Domains stacked out of set order: row group g must read AND write (dgamma / dbeta, running buffers) set int(domains[g]), not set g.
DOMS = [2, 0, 3, 1]


def _batches(dev, seed):
    return [tuple(t.to(dev) for t in synth.synth_batch(seed, d, 2, 64, 64)) + (d,) for d in DOMS]


def _trainer_step(dev, kind, am, fuse):
    from mdvit_b200.train_step import MKDTrainer
    m = _dsn(dev, kind, am).train()
    tr = MKDTrainer(m, with_aux=(kind == "mdvit"), fuse_domains=fuse)
    batches = _batches(dev, 1)
    tr.grad.zero_()
    losses = tr.forward_losses(batches)
    tr.backward(losses)
    torch.cuda.synchronize()
    bufs = {k: v.clone() for k, v in m.state_dict().items() if "running" in k or k.endswith("num_batches_tracked")}
    return losses.detach().clone(), {n: p.grad.detach().clone() for n, p in m.named_parameters()}, bufs


@pytest.mark.gpu
@pytest.mark.parametrize("kind,am", CASES)
def test_dsn_fused_trainer_step_equals_per_domain_step(env, kind, am):
    """MKDTrainer(fuse_domains=True) takes the stacked path for both DSN models (BASE_DSN through with_aux=False) and matches the
    per-domain loop: losses, gradients of every parameter (each domain's norm set gets its gradient from its own group only)
    and the BatchNorm buffers."""
    from mdvit_b200.train_step import MKDTrainer
    _, _, dev = env
    called = []
    m = _dsn(dev, kind, am)
    orig = m.forward_multi
    m.forward_multi = lambda *a: called.append(1) or orig(*a)
    tr = MKDTrainer(m, with_aux=(kind == "mdvit"))
    tr.forward_losses(_batches(dev, 1))
    assert called, "the fused trainer path was not taken"
    l0, g0, b0 = _trainer_step(dev, kind, am, False)
    l1, g1, b1 = _trainer_step(dev, kind, am, True)
    assert (l0 - l1).abs().max().item() < 5e-3 * l0.abs().max().item()
    g_all, w_tight, w_loose, text = grad_report(g1, g0, loose=("domain_layer", "bridge"))
    assert g_all < 0.02 and w_tight < 0.08 and w_loose < 0.12, text
    assert all(g1[n].abs().max().item() > 0 for n in g1 if ".norm1s." in n and n.endswith("weight")), "a norm set got no gradient"
    for k in b0:
        if k.endswith("num_batches_tracked"):
            assert int(b0[k]) == int(b1[k]) == 1, k
        else:
            assert rel(b1[k], b0[k]) < 5e-3, k


@pytest.mark.gpu
@pytest.mark.parametrize("kind,am", [("mdvit", "Sup"), ("base", None)])
def test_dsn_graph_step_equals_eager_step(env, kind, am):
    """The captured fused step (one CUDA graph; the per-group pointer tables are baked into its kernel parameters) follows the
    eager trainer over two optimizer steps."""
    from mdvit_b200.train_step import MKDTrainer
    _, _, dev = env
    batches = _batches(dev, 5)
    eager = MKDTrainer(_dsn(dev, kind, am).train(), with_aux=(kind == "mdvit"))
    graph = MKDTrainer(_dsn(dev, kind, am).train(), with_aux=(kind == "mdvit"))
    graph.capture(batches, warmup=2)
    l_eager = [eager.step(batches).clone() for _ in range(2)]
    l_graph = [graph.step_graph(None).clone() for _ in range(2)]
    torch.cuda.synchronize()
    assert graph.t == 2 and eager.t == 2
    for a, b in zip(l_eager, l_graph):
        assert (a - b).abs().max().item() < 2e-2 * a.abs().max().item()
    sd_e, sd_g = eager.model.state_dict(), graph.model.state_dict()
    for k in sd_e:
        if k.endswith("num_batches_tracked"):
            assert int(sd_e[k]) == int(sd_g[k]) == 2, k
