"""The trainer core MKDTrainer and TransFuseTrainer share (mdvit_b200/train_step.py): flat parameter / gradient buffers, the
device-side AdamW hyper-parameters, the domain-label rule of MKDTrainer's two forward paths (CPU, no kernels), and the input
staging rule of step_graph() on a captured step (GPU)."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from mdvit_b200 import ops
from mdvit_b200.train_step import MKDTrainer, TransFuseTrainer

TRAINERS = {"mkd": MKDTrainer, "transfuse": TransFuseTrainer}


class _Tiny(nn.Module):
    def __init__(self):
        super().__init__()
        self.a = nn.Linear(3, 5)                 # 15 + 5 elements: not multiples of 4
        self.b = nn.Conv2d(5, 7, 3)
        self.tied = nn.Linear(3, 5)
        self.tied.weight = self.a.weight         # a parameter shared by two modules gets one range of the flat buffer


@pytest.mark.parametrize("kind", sorted(TRAINERS))
def test_parameters_and_gradients_are_aligned_views_into_the_flat_buffers(kind):
    torch.manual_seed(0)
    m = _Tiny()
    before = {n: p.detach().clone() for n, p in m.named_parameters()}
    tr = TRAINERS[kind](m)
    assert len(tr.params) == len(before) == 5
    ends = []
    for n, p in m.named_parameters():
        o = p.data.storage_offset()
        assert o % 4 == 0, n
        assert p.data.untyped_storage().data_ptr() == tr.flat.untyped_storage().data_ptr(), n
        assert p.grad.untyped_storage().data_ptr() == tr.grad.untyped_storage().data_ptr() and p.grad.storage_offset() == o, n
        assert torch.equal(tr.flat[o:o + p.numel()], before[n].reshape(-1)) and torch.equal(p.detach(), before[n]), n
        ends.append((o, o + p.numel()))
    ends.sort()
    assert all(a[1] <= b[0] for a, b in zip(ends, ends[1:])) and ends[-1][1] <= tr.total == tr.flat.numel() == tr.grad.numel()


@pytest.mark.parametrize("kind", sorted(TRAINERS))
def test_lr_setter_writes_the_device_hyper_parameters(kind):
    tr = TRAINERS[kind](_Tiny(), lr=1e-4)
    assert tr.lr == 1e-4 and tr.hyper[0].item() == 1e-4 and tr.t == 0
    tr.lr = 0.25
    assert tr.lr == 0.25 and tr.hyper[0].item() == 0.25


@pytest.mark.parametrize("kind", sorted(TRAINERS))
def test_graph_replay_before_capture_raises(kind):
    tr = TRAINERS[kind](_Tiny())
    with pytest.raises(RuntimeError, match="capture"):
        tr.step_graph()
    with pytest.raises(RuntimeError, match="capture"):
        tr.prefetch([])


class _Recorder(nn.Module):
    """Stands in for MDViT / BASE / BASE_DSN: records the domain label of every call."""

    def __init__(self, aux, dsn, adapters, decoder):
        super().__init__()
        self.w = nn.Parameter(torch.ones(1))
        if adapters:
            self.domain_layer = nn.Linear(4, 2)
        if dsn:
            self.domain_specific_norms = True
        self.decoder_name = decoder
        self.aux, self.calls = aux, []

    def forward(self, x, domain_label=None, d=None):
        self.calls.append(domain_label)
        o = self.w * x[:, :1]
        return [o, o] if self.aux else o

    def forward_multi(self, x, domain_label, domains):
        self.calls.append(domain_label)
        return [(o, o if self.aux else None) for o in (self.w * x[:, :1]).chunk(len(domains))]


LABEL_CASES = {      # (with_aux, domain_specific_norms, domain adapters, decoder_name), and whether the model gets a label
    "mdvit": ((True, False, True, "MLPFM"), True),
    "base": ((False, False, False, None), False),
    "base_dsn_adapters": ((False, True, True, None), True),
    "base_dsn": ((False, True, False, None), False),
}


@pytest.mark.parametrize("case", sorted(LABEL_CASES))
def test_mkd_fused_and_per_domain_forwards_pass_the_same_domain_label(monkeypatch, case):
    (aux, dsn, adapters, decoder), labelled = LABEL_CASES[case]
    monkeypatch.setattr(ops, "seg_losses_multi", lambda outs, auxs, labels, **kw: torch.zeros(len(outs), 3))
    doms = [2, 0, 3]
    batches = [(torch.randn(2, 3, 8, 8), torch.zeros(2, 1, 8, 8), d) for d in doms]
    calls = {}
    for fused in (True, False):
        m = _Recorder(aux, dsn, adapters, decoder)
        MKDTrainer(m, with_aux=aux, fuse_domains=fused).forward_losses(batches)
        calls[fused] = m.calls
    assert len(calls[True]) == 1 and len(calls[False]) == len(doms)      # the fused path was taken, and the loop
    if not labelled:
        assert calls[True][0] is None and all(dl is None for dl in calls[False])
        return
    want = F.one_hot(torch.tensor(doms).repeat_interleave(2), 4).float()
    assert torch.equal(calls[True][0], want) and torch.equal(torch.cat(calls[False]), want)


# ------------------------------------------------------------------------------------------------- captured step (GPU)
def _mdvit(dev):
    from mdvit_b200 import synth
    from mdvit_b200.model import MDViT
    m = MDViT(img_size=64, adapt_method="Sup", num_domains=4, decoder_name="MLPFM").to(dev)
    m.load_state_dict(synth.synth_state_dict(0), strict=True)
    for k in range(1, 5):
        getattr(m, f"debranch{k}").dropout.p = 0.0
    return m.train()


def _transfuse(dev):
    from mdvit_b200.transfuse import TransFuse_S_adapt
    torch.manual_seed(0)
    return TransFuse_S_adapt(drop_rate=0.0).to(dev).train()


GRAPH_CASES = {"mkd": (MKDTrainer, _mdvit, 4, 64), "transfuse": (TransFuseTrainer, _transfuse, 2, 256)}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", sorted(GRAPH_CASES))
def test_prefetched_and_direct_replays_agree(kind):
    """Two identical captured trainers, one fed by prefetch() + step_graph(), the other by step_graph(batches): same inputs, so
    the same losses and weights up to the fp32 reduce-add order of the weight gradients (tolerances of the eager-versus-graph
    tests).  Then on the captured step: step_graph(batches) with a prefetch pending raises, and a replay at lr = 0 leaves the
    weights unchanged while the step count advances (the graph reads the trainer's device hyper-parameters)."""
    from mdvit_b200 import synth
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dev = torch.device("cuda")
    cls, build, G, side = GRAPH_CASES[kind]
    host = []      # two steps' inputs in pinned host memory
    for seed in (5, 6):
        batches = [synth.synth_batch(seed, d, 2, side, side) for d in range(G)]
        host.append([(img.pin_memory(), lab.to(torch.uint8).pin_memory(), d) for d, (img, lab) in enumerate(batches)])
    runs = []
    for prefetched in (True, False):
        ops.manual_seed(7, dev)
        tr = cls(build(dev), lr=1e-3, weight_decay=0.0)
        p0 = tr.flat.clone()
        tr.capture([(i.to(dev), l.to(dev), d) for i, l, d in host[0]], warmup=1)
        if prefetched:
            tr.prefetch(host[0])
            tr.prefetch(host[1])
            ls = [tr.step_graph().clone() for _ in range(2)]
        else:
            ls = [tr.step_graph(b).clone() for b in host]
        torch.cuda.synchronize()
        assert tr.t == 2
        assert all(torch.equal(s[0].cpu(), h[0]) and torch.equal(s[1].cpu(), h[1]) for s, h in zip(tr.static, host[1]))
        runs.append((torch.stack(ls).cpu(), tr.flat.clone(), p0, tr))
    (l0, f0, p0, tr), (l1, f1, _, _) = runs
    assert torch.isfinite(l0).all() and not torch.equal(l0[0], l0[1])
    if kind == "mkd":
        assert (l0 - l1).abs().max().item() < 2e-2 * l0.abs().max().item(), (l0, l1)
    else:
        assert torch.allclose(l0, l1, rtol=2e-3), (l0, l1)
    assert (f0 - p0).abs().max().item() > 0.5e-3
    diff = (f0 - f1).abs()
    assert diff.median().item() < 5e-5 and (diff > 5e-4).float().mean().item() < 2e-2, (diff.median().item(), (diff > 5e-4).float().mean().item())

    tr.prefetch(host[0])
    with pytest.raises(RuntimeError, match="prefetch"):
        tr.step_graph(host[1])
    tr.step_graph()
    tr.lr = 0.0
    before = tr.flat.clone()
    tr.step_graph()
    torch.cuda.synchronize()
    assert tr.t == 4 and torch.equal(tr.flat, before)
