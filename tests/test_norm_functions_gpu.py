"""The MDViT norm Functions (ops.StemFn, PatchEmbedFn, BlockFn, BridgeFn, DecoderConvFn, HeadFn) called directly, against a float64
restatement built from oracle/mdvit_oracle.py and run on the same GPU (TF32 off, gradients from torch autograd).

Every Function runs on non-square maps, down to the 1x1 / 1x2 deepest maps of the smallest legal images (32x32, 32x64), and in each
norm mode it has:
  train1        train mode, one norm set;
  train_shared  train mode, G stacked mini-batches sharing one set (ops.bn_groups(G)): the reference is G consecutive BatchNorm
                calls on the row slices, so the running buffers update in group order and num_batches_tracked grows by G;
  train_sets    train mode, G stacked mini-batches with G distinct sets (the domain-specific-norm path): slice g uses set g;
  eval1         eval mode, one set (BatchNorm folded into the GEMM epilogue);
  eval_sets     eval mode inside ops.norm_sets(idx) with 3 distinct sets and an unsorted per-sample index vector.
Distinct sets come from synth.dsn_perturb, so a kernel reading the wrong set, the wrong slot or the wrong sample shows.  The loss is
sum(y * R) for a fixed random probe R; the output, every input and parameter gradient (each norm set's included) and every set's
running_mean / running_var / num_batches_tracked are compared.

Bounds (TOL below) are about 3x the largest error measured over all cases of a Function on one B200; the measured values are written
next to them.  Forward errors are max|y - ref| / max|ref|; gradient errors are relative L2, with the "fraction of large deviations"
guard of test_transfuse_model_gpu._conv_case against activation-mask flips.  The conv biases in front of the bridge's train-mode
BatchNorms have an exactly-zero true gradient and are compared on an absolute scale (against the largest weight-gradient norm of
the Function).  The bridge's gradient bounds (0.115 / 0.19) are above the model-level loose class (0.12) for bridge.*: its cases
normalise 12-45 rows per group (the model tests at 64x64 normalise 32), and the bf16 input-gradient GEMMs (K = 9 x 512) feed that
BatchNorm's backward, whose cancellation grows as the rows get fewer.
"""
import contextlib
import functools
import math
import zlib

import pytest
import torch
import torch.nn.functional as F

from mdvit_b200 import ops, synth
from oracle import mdvit_oracle as O

pytestmark = pytest.mark.gpu

F64 = torch.float64
BN_BUFS = ("running_mean", "running_var", "num_batches_tracked")

# per Function: out = forward, dx = input gradients, dw = weight / bias gradients, dn = norm-parameter gradients,
# buf = running buffers (max-abs relative), zero = gradients that are exactly zero in exact arithmetic (absolute scale)
TOL = {      # measured maxima on one B200 (1000 W power limit) in the comments
    "stem": dict(out=6e-3, dw=2.5e-2, dn=3.5e-2, buf=1e-3),                           # 2.1e-3 7.2e-3 1.2e-2 3.5e-4
    "patch": dict(out=4e-3, dx=1.3e-2, dw=1.5e-2, dn=4e-2, buf=5e-4),                 # 1.2e-3 4.2e-3 4.7e-3 1.4e-2 1.7e-4
    "block": dict(out=1.2e-2, dx=1.2e-2, dw=2.2e-2, dn=2.1e-2),                       # 3.9e-3 3.8e-3 7.3e-3 7.0e-3
    "bridge": dict(out=4e-3, dx=0.115, dw=0.115, dn=0.19, buf=1.3e-3, zero=1.5e-4),   # 1.3e-3 3.8e-2 3.9e-2 6.4e-2 4.1e-4 4.9e-5
    "decoder": dict(out=4.5e-3, dx=1.7e-2, dw=2.6e-2, dn=3.8e-2, buf=1e-3),           # 1.5e-3 5.5e-3 8.5e-3 1.3e-2 3.4e-4
    "head": dict(out=5e-7, dx=3e-7, dw=1.2e-6),                                       # 1.6e-7 8.2e-8 4.0e-7 (fp32 throughout)
    "patch_few": dict(out=5e-2, dx=3.5e-2, dw=3.5e-2, dn=4e-3, buf=5e-4),             # 1.5e-2 1.1e-2 1.2e-2 1.2e-3 1.7e-4
    "bridge_few": dict(out=0.3, buf=2e-3, zero=2.5e-4),                               # 9.8e-2 6.4e-4 8.2e-5
    "decoder_few": dict(out=7e-2, dx=7.5e-2, dw=7.5e-2, dn=1e-2, buf=1e-3),           # 2.4e-2 2.5e-2 2.5e-2 2.8e-3 3.3e-4
}
# Fewer rows than this per channel and group make a train-mode BatchNorm ill-conditioned: with n rows, y = (z - mean) / sqrt(var + eps)
# amplifies the TF32 rounding of z where the rows nearly agree, and for n = 2 the outputs are +-1 whatever z is, so the exact gradient
# upstream of the BatchNorm is zero and what a comparison would see is round-off (measured relative L2 1.1 for the bridge's input and
# conv weights at 1x2 with one sample per group).  Those cases (the bridge at 1x1 / 1x2 / 2x2, the last patch embedding at 1x1,
# decoder1 at 1x2) get the *_few bounds, which are looser than the model-level bounds for the same reason: the model tests never
# normalise fewer than 8 rows.  Gradient kinds missing from a *_few entry (the bridge's) are only checked to be finite.
FEW_ROWS = 8
# ReLU / Hardswish mask flips: at most 0.6 % of a gradient's entries may be off by 0.1 of its abs-max (5x the op-level 2e-2); measured
# 0.2 % (2 of the 1024 entries of bridge.4.bias at 2x2)
BIG_DEV, BIG_FRAC = 0.1, 6e-3


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return torch.device("cuda")


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return ((a - b).abs().max() / (b.abs().max() + 1e-30)).item()


def rel_l2(a, b):
    a, b = a.detach().double(), b.detach().double()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def _tok(x):
    """NCHW -> token-major [B, H*W, C]."""
    return x.flatten(2).transpose(1, 2)


def _img(t, H, W):
    """token-major [B, H*W, C] -> NCHW."""
    return t.transpose(1, 2).reshape(t.shape[0], t.shape[2], H, W)


@functools.lru_cache(maxsize=1)
def _synth():
    return synth.synth_state_dict(0)


def _norm_set(prefix, s, S, bn):
    """Set s of the norm whose MDViT state-dict prefix is `prefix`: the synth values when there is one set; synth.dsn_perturb's values
    (keyed by set) when there are several, so that the sets really differ."""
    sd = _synth()
    vals = {leaf: sd[f"{prefix}.{leaf}"] for leaf in ("weight", "bias") + (BN_BUFS if bn else ())}
    if S == 1:
        return {k: v.clone() for k, v in vals.items()}
    tag = "bns" if bn else "norm1s"
    out = synth.dsn_perturb({f"{prefix}.{tag}.{s}.{leaf}": v for leaf, v in vals.items()})
    return {k.rsplit(".", 1)[1]: v for k, v in out.items()}


# ------------------------------------------------------------------------------------------------- reference pieces
def bridge_ref(sd, x, training):
    """bridge, mdvit.py:557-564 (as in mdvit_oracle.mdvit_forward): 2x (Conv3x3 + bias -> BatchNorm -> ReLU)."""
    out = F.conv2d(x, sd["bridge.0.weight"], sd["bridge.0.bias"], padding=1)
    out = F.relu(O.batchnorm(sd, "bridge.1", out, training))
    out = F.conv2d(out, sd["bridge.3.weight"], sd["bridge.3.bias"], padding=1)
    return F.relu(O.batchnorm(sd, "bridge.4", out, training))


def decoder_conv_ref(sd, prefix, x, skip, training):
    """The conv part of UnetDecodingBlockTransformer.forward, Decoders.py:194-205 (mdvit_oracle.decoder_block before its MHSA
    stage): bilinear resize to the skip's size -> 1x1 conv_before -> cat(skip, .) -> grouped 3x3 -> 1x1 -> BatchNorm -> Hardswish."""
    H, W = skip.shape[2:]
    out = O.bilinear(x, (H, W))
    out = F.conv2d(out, sd[prefix + ".conv_before.weight"], sd[prefix + ".conv_before.bias"])
    out = torch.cat((skip, out), dim=1)
    out = F.conv2d(out, sd[prefix + ".conv_after.dwconv.weight"], None, padding=1, groups=skip.shape[1])
    out = F.conv2d(out, sd[prefix + ".conv_after.pwconv.weight"], None)
    return O.hardswish(O.batchnorm(sd, prefix + ".conv_after.bn", out, training))


def head_ref(sd, x, size):
    """mdvit.py:699-700: bilinear resize to the image size -> finalconv (1x1, C -> 1)."""
    return F.conv2d(O.bilinear(x, size), sd["finalconv.0.weight"], sd["finalconv.0.bias"])


# ------------------------------------------------------------------------------------------------- the Functions
# Each spec: weights = state-dict keys of the Function's non-norm parameters in argument order (None: argument passed as None);
# norms = prefixes of its norm slots in order; bn = whether they are BatchNorms; inputs(B, g) = [(tensor, differentiable)];
# impl(xs, ws, norm, bufs, training) calls the Function; ref(sd, xs, training) is the float64 restatement on one group's slice.
def stem_spec(H, W):
    def inputs(B, g):
        return [(torch.randn((B, 3, H, W), generator=g), False)]

    def impl(xs, ws, norm, bufs, training):
        return ops.StemFn.apply(xs[0], ws[0], ws[1], bufs, training, *norm)

    def ref(sd, xs, training):      # mdvit.py:509-526, 667
        y = O.conv_bn_act(sd, "stem.0", xs[0], 2, 1, training, O.hardswish)
        return _tok(O.conv_bn_act(sd, "stem.1", y, 2, 1, training, O.hardswish))

    return dict(fn="stem", weights=["stem.0.conv.weight", "stem.1.conv.weight"], norms=["stem.0.bn", "stem.1.bn"], bn=True,
                inputs=inputs, impl=impl, ref=ref, areas=[H * W // 4, H * W // 16])


def patch_spec(i, Hi, Wi, after_stem):
    Cin, C, s = (synth.EMBED[i - 1] if i else synth.EMBED[0]), synth.EMBED[i], (1 if i == 0 else 2)
    Ho, Wo = (Hi - 1) // s + 1, (Wi - 1) // s + 1
    p = f"patch_embed_stages.{i}"

    def inputs(B, g):
        return [(torch.randn((B, Hi * Wi, Cin), generator=g), True)]

    def impl(xs, ws, norm, bufs, training):
        return ops.PatchEmbedFn.apply(xs[0], ws[0], ws[1], bufs, Hi, Wi, s, training, after_stem, *norm)

    def ref(sd, xs, training):
        return _tok(O.patch_embed(sd, p, _img(xs[0], Hi, Wi), s, training))

    return dict(fn="patch", weights=[p + ".patch_conv.dwconv.weight", p + ".patch_conv.pwconv.weight"], norms=[p + ".patch_conv.bn"],
                bn=True, inputs=inputs, impl=impl, ref=ref, areas=[Ho * Wo])


def block_spec(C, H, W, sup):
    i = synth.EMBED.index(C)
    st = f"mhsa_stages.{i}"
    blk, a = f"{st}.mhca_blks.0", f"{st}.mhca_blks.0.factoratt_crpe"
    da = [f"{a}.domain_layer.{j}.{t}" for j in (0, 2) for t in ("weight", "bias")] if sup else [None] * 4

    def inputs(B, g):
        label = F.one_hot(torch.randint(0, 4, (B,), generator=g), 4).float()
        return [(torch.randn((B, H * W, C), generator=g), True), (label, False)]

    def impl(xs, ws, norm, bufs, training):
        return ops.BlockFn.apply(xs[0], xs[1] if sup else None, *ws, H, W, 0.0, 0.0, training, *norm)

    def ref(sd, xs, training):      # drop = dpr = 0
        return O.serial_block(sd, st, 0, xs[0], H, W, xs[1] if sup else None, training=training)

    weights = ([f"{st}.cpe.proj.weight", f"{st}.cpe.proj.bias"] + [f"{st}.crpe.conv_list.{j}.{t}" for j in range(3) for t in ("weight", "bias")]
               + [f"{a}.qkv.weight", f"{a}.qkv.bias", f"{a}.proj.weight", f"{a}.proj.bias"] + da
               + [f"{blk}.mlp.fc1.weight", f"{blk}.mlp.fc1.bias", f"{blk}.mlp.fc2.weight", f"{blk}.mlp.fc2.bias"])
    return dict(fn="block", weights=weights, norms=[blk + ".norm1", blk + ".norm2"], bn=False, inputs=inputs, impl=impl, ref=ref,
                areas=[])


def bridge_spec(H, W):
    def inputs(B, g):
        return [(torch.randn((B, H * W, 512), generator=g), True)]

    def impl(xs, ws, norm, bufs, training):
        return ops.BridgeFn.apply(xs[0], *ws, bufs, H, W, training, *norm)

    def ref(sd, xs, training):
        return _tok(bridge_ref(sd, _img(xs[0], H, W), training))

    return dict(fn="bridge", weights=["bridge.0.weight", "bridge.0.bias", "bridge.3.weight", "bridge.3.bias"], norms=["bridge.1", "bridge.4"],
                bn=True, inputs=inputs, impl=impl, ref=ref, areas=[H * W, H * W], zero_grad=["bridge.0.bias", "bridge.3.bias"])


def decoder_spec(k, h, w, H, W):
    Cin, C = ((1024, 512), (512, 320), (320, 128), (128, 64))[k - 1]
    p = f"decoder{k}"

    def inputs(B, g):
        return [(torch.randn((B, h * w, Cin), generator=g), True), (torch.randn((B, H * W, C), generator=g), True)]

    def impl(xs, ws, norm, bufs, training):
        return ops.DecoderConvFn.apply(xs[0], xs[1], *ws, bufs, h, w, H, W, training, *norm)

    def ref(sd, xs, training):
        return _tok(decoder_conv_ref(sd, p, _img(xs[0], h, w), _img(xs[1], H, W), training))

    return dict(fn="decoder", weights=[p + ".conv_before.weight", p + ".conv_before.bias", p + ".conv_after.dwconv.weight",
                                       p + ".conv_after.pwconv.weight"],
                norms=[p + ".conv_after.bn"], bn=True, inputs=inputs, impl=impl, ref=ref, areas=[H * W])


def head_spec(H, W, Ho, Wo):
    def inputs(B, g):
        return [(torch.randn((B, H * W, 64), generator=g), True)]

    def impl(xs, ws, norm, bufs, training):
        return ops.HeadFn.apply(xs[0], ws[0], ws[1], H, W, Ho, Wo)

    def ref(sd, xs, training):
        return head_ref(sd, _img(xs[0], H, W), (Ho, Wo))

    return dict(fn="head", weights=["finalconv.0.weight", "finalconv.0.bias"], norms=[], bn=False, inputs=inputs, impl=impl, ref=ref,
                areas=[])


# ------------------------------------------------------------------------------------------------- cases
MODES = ("train1", "train_shared", "train_sets", "eval1", "eval_sets")
SAMPLE_SETS = {1: [1], 2: [1, 0], 3: [2, 0, 1], 4: [2, 0, 1, 0]}      # per-sample set indices: not sorted, not constant (S = 3)


def _groups(B, areas):
    """G of the stacked modes: every group holds whole samples and every BatchNorm sees at least 2 rows per group (nn.BatchNorm2d
    rejects a single value per channel in training).  None: no stacked mode for this batch."""
    for G in (3, 2):
        if B % G == 0 and all(B // G * a >= 2 for a in areas):
            return G
    return None


def _cases():
    specs = []
    for H, W in ((64, 64), (96, 160), (160, 96), (32, 64)):
        for B in (1, 3):
            specs.append((f"stem-{H}x{W}-B{B}", ("stem", H, W), B))
    for i, Hi, Wi, after in ((0, 24, 40, True), (0, 24, 40, False), (1, 24, 40, False), (2, 12, 20, False), (3, 6, 10, False),
                             (3, 2, 2, False)):
        B = 4 if Hi == 2 else 3
        specs.append((f"patch{i}-{Hi}x{Wi}{'-after_stem' if after else ''}-B{B}", ("patch", i, Hi, Wi, after), B))
    for C, H, W in ((64, 24, 40), (128, 12, 20), (320, 6, 10), (512, 3, 5), (320, 2, 2), (512, 1, 1), (512, 1, 2)):
        for sup in (True, False):
            specs.append((f"block{C}-{H}x{W}-{'sup' if sup else 'plain'}-B3", ("block", C, H, W, sup), 3))
    for H, W, B in ((1, 1, 1), (1, 1, 3), (1, 2, 1), (1, 2, 3), (3, 5, 1), (3, 5, 3), (2, 2, 3)):
        specs.append((f"bridge-{H}x{W}-B{B}", ("bridge", H, W), B))
    for k, h, w, H, W in ((1, 3, 5, 3, 5), (1, 1, 2, 1, 2), (2, 3, 5, 6, 10), (2, 1, 2, 2, 4), (3, 6, 10, 12, 20), (3, 10, 6, 20, 12),
                          (4, 12, 20, 24, 40)):
        specs.append((f"decoder{k}-{h}x{w}-{H}x{W}-B3", ("decoder", k, h, w, H, W), 3))
    for H, W, Ho, Wo in ((24, 40, 96, 160), (40, 24, 160, 96)):
        specs.append((f"head-{H}x{W}-{Ho}x{Wo}-B2", ("head", H, W, Ho, Wo), 2))
    out = []
    for name, geo, B in specs:
        spec = _spec(geo)
        for mode in MODES:
            if not spec["norms"] and mode != "train1":
                continue
            if not spec["bn"] and mode == "train_shared":      # LayerNorm has no batch statistics: the same as train1
                continue
            if mode.startswith("train") and any(B * a < 2 for a in spec["areas"]):
                continue
            if mode in ("train_shared", "train_sets") and _groups(B, spec["areas"]) is None:
                continue
            out.append(pytest.param(geo, B, mode, id=f"{name}-{mode}"))
    return out


def _spec(geo):
    return {"stem": stem_spec, "patch": patch_spec, "block": block_spec, "bridge": bridge_spec, "decoder": decoder_spec,
            "head": head_spec}[geo[0]](*geo[1:])


def _leaf(t, dev, dtype):
    return t.to(dev, dtype).clone().requires_grad_(True)


def _grad_err(what, kind, got, want, report, guard):
    """Relative L2 error of a gradient, and (guard) the share of entries off by more than BIG_DEV of max|want|."""
    assert got is not None, f"{what}: no gradient"
    report.append((what, kind, rel_l2(got, want)))
    if guard:
        big = ((got.double() - want.double()).abs() > BIG_DEV * want.double().abs().max()).double().mean().item()
        report.append((what, "big", big))


@pytest.mark.parametrize("geo,B,mode", _cases())
def test_norm_function_vs_fp64(dev, geo, B, mode):
    spec = _spec(geo)
    training = mode.startswith("train")
    k = len(spec["norms"])
    G = _groups(B, spec["areas"]) if mode in ("train_shared", "train_sets") else 1
    S = {"train_sets": G, "eval_sets": 3}.get(mode, 1) if k else 1
    idx = SAMPLE_SETS[B] if mode == "eval_sets" else None
    g = torch.Generator().manual_seed(zlib.crc32(repr((geo, B, mode)).encode()))
    xs = spec["inputs"](B, g)
    sd = _synth()
    sets = [[_norm_set(p, s, S, spec["bn"]) for p in spec["norms"]] for s in range(S)]

    # ---- the Function (fp32 inputs and parameters)
    x32 = [x.to(dev).requires_grad_(d and training) for x, d in xs]
    w32 = [None if key is None else _leaf(sd[key], dev, torch.float32) for key in spec["weights"]]
    n32 = [[{leaf: _leaf(st[leaf], dev, torch.float32) for leaf in ("weight", "bias")} for st in slots] for slots in sets]
    b32 = [[{leaf: st[leaf].to(dev).clone() for leaf in BN_BUFS} for st in slots] for slots in sets] if spec["bn"] else []
    norm = tuple(t for slots in n32 for st in slots for t in (st["weight"], st["bias"]))
    bufs = tuple(t for slots in b32 for st in slots for t in (st["running_mean"], st["running_var"], st["num_batches_tracked"]))
    if mode == "eval_sets":
        ctx = ops.norm_sets(torch.tensor(idx, dtype=torch.int32, device=dev))
    elif mode in ("train_shared", "train_sets"):
        ctx = ops.bn_groups(G)
    else:
        ctx = contextlib.nullcontext()
    with ctx, torch.set_grad_enabled(training):
        y = spec["impl"](x32, w32, norm, bufs, training)
    probe = torch.randn(tuple(y.shape), generator=g).to(dev)
    if training:
        (y * probe).sum().backward()
    torch.cuda.synchronize()

    # ---- the float64 reference, one call per row group (per sample in eval_sets)
    x64 = [x.to(dev, F64).requires_grad_(d and training) for x, d in xs]
    w64 = {key: _leaf(sd[key], dev, F64) for key in spec["weights"] if key is not None}
    sds = []
    for s in range(S):
        d = dict(w64)
        for j, p in enumerate(spec["norms"]):
            d[p + ".weight"], d[p + ".bias"] = (_leaf(sets[s][j][leaf], dev, F64) for leaf in ("weight", "bias"))
            if spec["bn"]:
                d[p + ".running_mean"], d[p + ".running_var"] = (sets[s][j][leaf].to(dev, F64).clone() for leaf in BN_BUFS[:2])
                d[p + ".num_batches_tracked"] = sets[s][j]["num_batches_tracked"].to(dev).clone()
        sds.append(d)
    if mode == "eval_sets":
        parts = [(sds[idx[b]], b, b + 1) for b in range(B)]
    else:
        n = B // G
        parts = [(sds[gi if S > 1 else 0], gi * n, (gi + 1) * n) for gi in range(G)]
    with torch.set_grad_enabled(training):
        ref = torch.cat([spec["ref"](d, [x[lo:hi] for x in x64], training) for d, lo, hi in parts])
    if training:
        (ref * probe.double()).sum().backward()

    # a train-mode BatchNorm over fewer than 8 rows per channel and group is ill-conditioned (see FEW_ROWS): its own bounds
    few = training and spec["bn"] and min(B // G * a for a in spec["areas"]) < FEW_ROWS
    tol = TOL[spec["fn"] + ("_few" if few else "")]
    report = [("y", "out", rel(y.reshape(ref.shape), ref))]
    if training:
        for i, ((x, d), a, r) in enumerate(zip(xs, x32, x64)):
            if d:
                _grad_err(f"dx{i}", "dx", a.grad, r.grad, report, not few)
        zero = spec.get("zero_grad", [])
        gmax = max(w64[key].grad.norm().item() for key in w64 if key not in zero)
        for key, a in zip(spec["weights"], w32):
            if key in zero:      # exactly zero through the train-mode BatchNorm it feeds: round-off only, on the largest gradient's scale
                report.append((key, "zero", (a.grad.double() - w64[key].grad).norm().item() / gmax))
            elif key is not None:
                _grad_err(key, "dw", a.grad, w64[key].grad, report, not few)
        for s in range(S):
            for j, p in enumerate(spec["norms"]):
                for leaf in ("weight", "bias"):
                    _grad_err(f"set{s}.{p}.{leaf}", "dn", n32[s][j][leaf].grad, sds[s][p + "." + leaf].grad, report, not few)
    if spec["bn"]:
        expect = {"train1": 1, "train_shared": G, "train_sets": 1}.get(mode, 0)
        for s in range(S):
            for j, p in enumerate(spec["norms"]):
                got, want = b32[s][j], sds[s]
                assert int(got["num_batches_tracked"]) == int(want[p + ".num_batches_tracked"]) == expect, (s, p)
                for leaf in BN_BUFS[:2]:
                    report.append((f"set{s}.{p}.{leaf}", "buf", rel(got[leaf], want[p + "." + leaf])))
                    if not training:
                        assert torch.equal(got[leaf].cpu(), sets[s][j][leaf]), "eval mode changed a running buffer"
    for what, kind, e in report:
        print(f"MEAS {spec['fn']}{'_few' if few else ''} {mode} {kind} {what} {e:.3e}")
    bad = [(what, kind, e) for what, kind, e in report if not (e < BIG_FRAC if kind == "big" else e < tol[kind] if kind in tol else math.isfinite(e))]
    assert not bad, bad


# ------------------------------------------------------------------------------------------------- whole model, non-square
def _f64_state_dict(dev):
    """The synth weights as a float64 oracle state_dict on the GPU: float leaves require grad, alias keys share their owner's tensor."""
    sd = {}
    for k, v in _synth().items():
        if synth.canonical_key(k) == k:
            t = v.to(dev, F64 if v.is_floating_point() else v.dtype).clone()
            sd[k] = t.requires_grad_(True) if t.is_floating_point() and "running" not in k else t
    for k in _synth():
        sd[k] = sd[synth.canonical_key(k)]
    return sd


@pytest.mark.parametrize("H,W", [(96, 160), (32, 64)])
def test_mdvit_non_square_vs_fp64(dev, H, W):
    """MDViT(adapt_method='Sup', decoder_name='MLPFM') on non-square images, B = 2, against mdvit_oracle.mdvit_forward in float64: the
    train-mode logits and aux logits, one backward's parameter gradients (bounds of
    test_model_gpu.test_train_step_losses_and_gradients_vs_reference_golden) and the eval logits after that step's BatchNorm
    updates.  32x64 makes the deepest map 1x2: the bridge normalises over 4 rows and the last stage attends over 2 tokens."""
    from tests.test_model_gpu import build, grad_report, onehot
    m = build(dev, H).train()
    sd = _f64_state_dict(dev)
    g = torch.Generator().manual_seed(H * 1000 + W)
    img = torch.randn((2, 3, H, W), generator=g).to(dev)
    dl = torch.stack([onehot(2, 1, dev)[0], onehot(0, 1, dev)[0]])
    probe = [torch.randn((2, 1, H, W), generator=g).to(dev) for _ in range(2)]
    out, aux = m(img, dl, "2")
    ro, ra = O.mdvit_forward(sd, img.double(), dl.double(), "2", training=True)
    report = [("out", rel(out, ro)), ("out_l2", rel_l2(out, ro)), ("aux", rel(aux, ra)), ("aux_l2", rel_l2(aux, ra))]
    ((out * probe[0]).sum() + (aux * probe[1]).sum()).backward()
    ((ro * probe[0].double()).sum() + (ra * probe[1].double()).sum()).backward()
    grads = {n: p.grad for n, p in m.named_parameters() if p.grad is not None}
    g_all, w_tight, w_loose, text = grad_report(grads, {n: sd[n].grad for n in grads})
    report += [("grad_all", g_all), ("grad_tight", w_tight), ("grad_loose", w_loose)]
    m.eval()
    with torch.no_grad():
        eo, ea = m(img, dl, "2")
        reo, rea = O.mdvit_forward(sd, img.double(), dl.double(), "2", training=False)
    report += [("eval_out", rel(eo, reo)), ("eval_out_l2", rel_l2(eo, reo)), ("eval_aux", rel(ea, rea)), ("eval_aux_l2", rel_l2(ea, rea))]
    for what, e in report:
        print(f"MEAS model {H}x{W} {what} {e:.3e}")
    assert out.shape == aux.shape == eo.shape == (2, 1, H, W)
    r = dict(report)
    # logits: measured <= 5.9e-3 (train), 7.8e-3 (eval) max-abs relative at both sizes, under the 2e-2 of test_model_gpu
    assert r["out"] < 2e-2 and r["out_l2"] < 2e-2 and r["aux"] < 2e-2 and r["aux_l2"] < 2e-2, report
    assert r["eval_out"] < 2.5e-2 and r["eval_out_l2"] < 2e-2 and r["eval_aux"] < 2e-2 and r["eval_aux_l2"] < 2e-2, report
    # gradients (global / worst tight / worst loose): measured 0.032 / 0.054 / 0.099 at 96x160, 0.105 / 0.213 / 0.182 at 32x64.  Under
    # this probe loss the largest gradient is bridge.0.weight's, whose path runs through the bridge's BatchNorms (30 rows per channel at
    # 96x160, 4 at 32x64: the ill-conditioned FEW_ROWS regime), so the global error sits above the 0.02 of the golden test; at 32x64
    # the 1x2 stage-3 maps (patch_embed 3 also normalises 4 rows) put every stage-3 tensor in the same regime.
    bound = (0.1, 0.16, 0.3) if H * W > 2048 else (0.32, 0.64, 0.55)
    assert g_all < bound[0] and w_tight < bound[1] and w_loose < bound[2], text
