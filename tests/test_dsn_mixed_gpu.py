"""MDViT_DSN / BASE_DSN inference on mixed-domain batches: the per-sample norm-set kernels (mdv_layernorm_fwd_sets,
mdv_gemm_nt_tf32_sets, mdv_bn_fold_sets) against torch and against their single-set counterparts, forward_mixed against
per-sample forwards, and a captured forward_mixed replayed on a new domain vector.  The models are loaded with
synth.dsn_perturb, so a kernel reading the wrong set would be visible."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from mdvit_b200 import synth

BF16_TOL = 1e-2


@pytest.fixture(scope="module")
def env():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    from mdvit_b200 import _lib as L
    return L, L.lib(), torch.device("cuda")


def rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-20)).item()


def _fake_table(addrs):
    from mdvit_b200 import _lib as L
    t = L.PtrTable()
    for i, a in enumerate(addrs):
        t.p[i] = a
    return t


# ------------------------------------------------------------------------------------------------- CPU: argument checks
def test_sets_entry_points_reject_bad_arguments(built_lib):
    """S outside 1..8, a missing table entry, a NULL sample_set / colscale and rows_per_sample < 1 return MDV_ERR_ARG (-1) before
    any CUDA call.  The pointers are never dereferenced."""
    from mdvit_b200 import _lib as L
    lib = built_lib
    p = [ctypes.c_void_p(0x10000 * (i + 1)) for i in range(8)]
    t = [_fake_table([0x100000 * (k + 1) + 0x1000 * g for g in range(8)]) for k in range(4)]
    e = L.GemmEpi()
    e.out, e.ldc, e.colscale, e.bias, e.act = p[5].value, 64, p[6].value, p[7].value, L.ACT_RELU
    for S in (0, 9):
        assert lib.mdv_layernorm_fwd_sets(p[0], t[0], t[1], 1e-6, p[1], None, None, p[2], 16, S, 64, 64, None) == -1
        assert lib.mdv_gemm_nt_tf32_sets(p[0], 64, p[1], 64, 64, 64, 64, ctypes.byref(e), p[2], 16, S, None) == -1
        assert lib.mdv_bn_fold_sets(t[0], t[1], t[2], t[3], None, 1e-5, p[3], p[4], S, 64, None) == -1
    # NULL sample_set, rows_per_sample < 1
    assert lib.mdv_layernorm_fwd_sets(p[0], t[0], t[1], 1e-6, p[1], None, None, None, 16, 2, 64, 64, None) == -1
    assert lib.mdv_layernorm_fwd_sets(p[0], t[0], t[1], 1e-6, p[1], None, None, p[2], 0, 2, 64, 64, None) == -1
    assert lib.mdv_gemm_nt_tf32_sets(p[0], 64, p[1], 64, 64, 64, 64, ctypes.byref(e), None, 16, 2, None) == -1
    assert lib.mdv_gemm_nt_tf32_sets(p[0], 64, p[1], 64, 64, 64, 64, ctypes.byref(e), p[2], 0, 2, None) == -1
    # NULL tables: a missing gamma / beta / buffer of a used set, a NULL colscale
    missing = _fake_table([0x500000])
    assert lib.mdv_layernorm_fwd_sets(p[0], missing, t[1], 1e-6, p[1], None, None, p[2], 16, 2, 64, 64, None) == -1
    assert lib.mdv_layernorm_fwd_sets(p[0], t[0], missing, 1e-6, p[1], None, None, p[2], 16, 2, 64, 64, None) == -1
    for k in range(4):
        tabs = [missing if j == k else t[j] for j in range(4)]
        assert lib.mdv_bn_fold_sets(*tabs, None, 1e-5, p[3], p[4], 2, 64, None) == -1
    e.colscale = None
    assert lib.mdv_gemm_nt_tf32_sets(p[0], 64, p[1], 64, 64, 64, 64, ctypes.byref(e), p[2], 16, 2, None) == -1


def test_forward_mixed_validates_before_any_launch(built_lib):
    """On a CPU-constructed model: train mode, a wrong number of keys, out-of-range or non-integer keys raise before any kernel
    launch (the launch counter does not move)."""
    from mdvit_b200.model import BASE_DSN, MDViT_DSN
    lib = built_lib
    n0 = lib.mdv_launch_count()
    for m in (MDViT_DSN(img_size=64, adapt_method="Sup", num_domains=4, decoder_name="MLPFM"), BASE_DSN(img_size=64, num_domains=4)):
        x = torch.zeros(3, 3, 64, 64)
        with pytest.raises(RuntimeError, match="forward_multi"):
            m.train().forward_mixed(x, None, [0, 1, 2])
        m.eval()
        with pytest.raises(ValueError):
            m.forward_mixed(x, None, [0, 1])                      # length
        with pytest.raises(ValueError):
            m.forward_mixed(x, None, torch.tensor([0, 1, 2, 3]))  # length (tensor)
        with pytest.raises(ValueError):
            m.forward_mixed(x, None, [0, 4, 1])                   # out of range
        with pytest.raises(ValueError):
            m.forward_mixed(x, None, ["0", "-1", "1"])
        with pytest.raises(ValueError):
            m.forward_mixed(x, None, torch.tensor([0, 1, 7]))
        with pytest.raises(TypeError):
            m.forward_mixed(x, None, [0, 1.5, 2])                 # not an integer key
        with pytest.raises(TypeError):
            m.forward_mixed(x, None, torch.tensor([0.0, 1.0, 2.0]))
    assert lib.mdv_launch_count() == n0


# ------------------------------------------------------------------------------------------------- kernels
@pytest.mark.gpu
@pytest.mark.parametrize("C", [64, 128, 320, 512])
@pytest.mark.parametrize("rps", [1, 16, 37])
def test_layernorm_fwd_sets_matches_torch_per_row(env, C, rps):
    """Row m normalised with set sample_set[m // rps] (random sets, S = 4) against torch fp32; mean / rstd NULL.  rps = 1 and 37
    put several samples into one warp's rows."""
    L, lib, dev = env
    torch.manual_seed(C + rps)
    S, B = 4, 29
    M = B * rps
    x = torch.randn(M, C, device=dev) * 2 + 0.5
    gs = [1 + 0.3 * torch.randn(C, device=dev) for _ in range(S)]
    bs = [0.3 * torch.randn(C, device=dev) for _ in range(S)]
    ss = torch.randint(0, S, (B,), device=dev, dtype=torch.int32)
    y = torch.empty(M, C, device=dev, dtype=torch.bfloat16)
    L.check(lib.mdv_layernorm_fwd_sets(L.ptr(x), L.ptr_table(gs), L.ptr_table(bs), 1e-6, L.ptr(y), None, None, L.ptr(ss), rps, S, M, C,
                                       L.stream()), "ln_sets")
    row_set = ss.long().repeat_interleave(rps)
    g, b = torch.stack(gs)[row_set], torch.stack(bs)[row_set]
    ref = F.layer_norm(x, (C,), eps=1e-6) * g + b
    assert rel(y, ref) < BF16_TOL
    # with mean / rstd requested they are the rows' statistics
    mean, rstd = torch.empty(M, device=dev), torch.empty(M, device=dev)
    L.check(lib.mdv_layernorm_fwd_sets(L.ptr(x), L.ptr_table(gs), L.ptr_table(bs), 1e-6, L.ptr(y), L.ptr(mean), L.ptr(rstd), L.ptr(ss), rps,
                                       S, M, C, L.stream()), "ln_sets")
    assert rel(mean, x.mean(1)) < 1e-5 and rel(rstd, (x.var(1, unbiased=False) + 1e-6).rsqrt()) < 1e-4


def tf32_representable(t):
    """round to 10 explicit mantissa bits: products of such operands are exact on the TF32 tensor cores and in fp32"""
    i = t.contiguous().view(torch.int32)
    return (((i + (1 << 12)) >> 13) << 13).view(torch.float32)


def _epi(L, out, N, scale, shift, act):
    e = L.GemmEpi()
    e.out, e.ldc, e.out_bf16, e.colscale, e.bias, e.act = L.ptr(out).value, N, 0, L.ptr(scale).value, L.ptr(shift).value, act
    return e


@pytest.mark.gpu
@pytest.mark.parametrize("pair", [0, 1])
@pytest.mark.parametrize("rps,B,N,K", [(64, 37, 512, 4608), (100, 13, 320, 64), (4096, 3, 64, 32), (64, 100, 64, 288)])
@pytest.mark.parametrize("act", [3, 2])
def test_gemm_nt_tf32_sets_matches_torch(env, rps, B, N, K, act, pair):
    """v = act(acc * colscale[s, n] + bias[s, n]) with s = sample_set[m // rows_per_sample], S = 5 random sets, against torch on
    TF32-representable operands.  M = B * rps is ragged for rps = 100 (M % 128 != 0) and rps = 64 puts two samples in one
    128-row tile; pairs forced on and off (16 epilogue warps: act is HSWISH or RELU)."""
    L, lib, dev = env
    torch.manual_seed(rps + B + N + K + act)
    S, M = 5, rps * B
    A = tf32_representable(torch.randn(M, K, device=dev))
    W = tf32_representable(torch.randn(N, K, device=dev) / K ** 0.5)
    sc = 1 + 0.3 * torch.randn(S, N, device=dev)
    sh = 0.3 * torch.randn(S, N, device=dev)
    ss = torch.randint(0, S, (B,), device=dev, dtype=torch.int32)
    rs = ss.long().repeat_interleave(rps)
    z = (A.double() @ W.double().t()) * sc.double()[rs] + sh.double()[rs]
    ref = (F.relu(z) if act == 2 else F.hardswish(z)).float()
    out = torch.full((M, N), float("nan"), device=dev)
    e = _epi(L, out, N, sc, sh, act)
    lib.mdv_gemm_force_pair(pair)
    try:
        L.check(lib.mdv_gemm_nt_tf32_sets(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(e), L.ptr(ss), rps, S, L.stream()), "gemm_sets")
    finally:
        lib.mdv_gemm_force_pair(-1)
    assert rel(out, ref) < 1e-4, pair       # (fp32 accumulation over K up to 4608 against fp64)


@pytest.mark.gpu
@pytest.mark.parametrize("pair", [-1, 0, 1])
@pytest.mark.parametrize("M,N,K,act", [(4096, 64, 32, 3), (1000, 320, 64, 3), (2048, 512, 4608, 2)])
def test_gemm_nt_tf32_sets_single_set_is_bit_identical(env, M, N, K, act, pair):
    """Every sample on set k: the sets GEMM equals mdv_gemm_nt_tf32 with set k's [N] tables bit for bit (same tiles, same epilogue
    arithmetic, only the table offset differs)."""
    L, lib, dev = env
    torch.manual_seed(M + N + K)
    S, rps = 4, 64
    A, W = torch.randn(M, K, device=dev), torch.randn(N, K, device=dev) / K ** 0.5
    sc, sh = 1 + 0.3 * torch.randn(S, N, device=dev), 0.3 * torch.randn(S, N, device=dev)
    lib.mdv_gemm_force_pair(pair)
    try:
        for k in (0, 3):
            ss = torch.full((-(-M // rps),), k, device=dev, dtype=torch.int32)
            o1, o2 = torch.empty(M, N, device=dev), torch.empty(M, N, device=dev)
            L.check(lib.mdv_gemm_nt_tf32_sets(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(_epi(L, o1, N, sc, sh, act)), L.ptr(ss), rps, S,
                                              L.stream()), "gemm_sets")
            s1, h1 = sc[k].clone(), sh[k].clone()
            L.check(lib.mdv_gemm_nt_tf32(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(_epi(L, o2, N, s1, h1, act)), L.stream()), "gemm")
            assert torch.equal(o1, o2), (k, pair)
    finally:
        lib.mdv_gemm_force_pair(-1)


@pytest.mark.gpu
@pytest.mark.parametrize("C,with_bias", [(32, False), (320, True), (1024, True)])
def test_bn_fold_sets_equals_per_set_bn_fold(env, C, with_bias):
    L, lib, dev = env
    torch.manual_seed(C)
    S = 6
    g, b = [1 + 0.3 * torch.randn(C, device=dev) for _ in range(S)], [0.3 * torch.randn(C, device=dev) for _ in range(S)]
    rm, rv = [0.2 * torch.randn(C, device=dev) for _ in range(S)], [1 + 0.3 * torch.rand(C, device=dev) for _ in range(S)]
    cb = torch.randn(C, device=dev) if with_bias else None
    sc, sh = torch.empty(S, C, device=dev), torch.empty(S, C, device=dev)
    L.check(lib.mdv_bn_fold_sets(L.ptr_table(g), L.ptr_table(b), L.ptr_table(rm), L.ptr_table(rv), L.ptr(cb), 1e-5, L.ptr(sc), L.ptr(sh), S,
                                 C, L.stream()), "bn_fold_sets")
    for k in range(S):
        s1, h1 = torch.empty(C, device=dev), torch.empty(C, device=dev)
        L.check(lib.mdv_bn_fold(L.ptr(g[k]), L.ptr(b[k]), L.ptr(rm[k]), L.ptr(rv[k]), L.ptr(cb), 1e-5, L.ptr(s1), L.ptr(h1), C, L.stream()),
                "bn_fold")
        assert torch.equal(sc[k], s1) and torch.equal(sh[k], h1), k


# ------------------------------------------------------------------------------------------------- models
_MODELS = {}


def _dsn(dev, kind, am):
    key = (kind, am)
    if key not in _MODELS:
        from mdvit_b200.model import BASE_DSN, MDViT_DSN
        torch.manual_seed(0)
        m = MDViT_DSN(img_size=64, adapt_method=am, num_domains=4, decoder_name="MLPFM") if kind == "mdvit" else \
            BASE_DSN(img_size=64, adapt_method=am, num_domains=4)
        m.load_state_dict(synth.dsn_perturb(m.state_dict()), strict=True)
        m.skip_aux_in_eval = True
        _MODELS[key] = m.to(dev).eval()
    return _MODELS[key]


def _main(m, x, dl, d):
    o = m(x, dl, d)
    return o[0] if isinstance(o, list) else o


def _inputs(dev, B, size, doms, am):
    x = torch.cat([synth.synth_batch(7 + i, d, 1, size, size)[0] for i, d in enumerate(doms)]).to(dev)
    dl = F.one_hot(torch.tensor(doms), 4).float().to(dev) if am else None
    return x, dl


@pytest.mark.gpu
@pytest.mark.parametrize("kind,am", [("mdvit", "Sup"), ("mdvit", None), ("base", "Sup"), ("base", None)])
@pytest.mark.parametrize("size", [64, 256])
@pytest.mark.parametrize("B", [1, 5, 8])
def test_forward_mixed_equals_per_sample_forwards(env, kind, am, size, B):
    """forward_mixed on domains not in set order against forward(x[i:i+1], dl[i:i+1], str(d_i)) per sample; a single-domain
    batch against forward(x, dl, d)."""
    _, _, dev = env
    m = _dsn(dev, kind, am)
    doms = [(3 * i + 2) % 4 for i in range(B)]
    x, dl = _inputs(dev, B, size, doms, am)
    with torch.no_grad():
        out = m.forward_mixed(x, dl, [str(d) for d in doms])
        assert out.shape == (B, 1, size, size)
        for i, d in enumerate(doms):
            ref = _main(m, x[i:i + 1], None if dl is None else dl[i:i + 1], str(d))
            assert rel(out[i:i + 1], ref) <= 1e-5, (i, d)
        d = 1
        dl1 = F.one_hot(torch.full((B,), d), 4).float().to(dev) if am else None
        out1 = m.forward_mixed(x, dl1, torch.full((B,), d))
        assert rel(out1, _main(m, x, dl1, str(d))) <= 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("kind,am", [("mdvit", "Sup"), ("base", None)])
def test_forward_mixed_graph_replays_new_domain_vector(env, kind, am):
    """Capture forward_mixed with a CUDA int32 domain tensor, write another domain vector into it, replay: the result equals the
    eager forward_mixed on that vector.  The mixed forward launches exactly as many library kernels as a single-domain eval
    forward with skip_aux_in_eval."""
    L, lib, dev = env
    m = _dsn(dev, kind, am)
    B, size = 6, 64
    doms_a, doms_b = [0, 1, 2, 3, 0, 1], [3, 3, 1, 0, 2, 1]
    x, _ = _inputs(dev, B, size, doms_a, am)
    dl = F.one_hot(torch.tensor(doms_b), 4).float().to(dev) if am else None
    dom_dev = torch.tensor(doms_a, dtype=torch.int32, device=dev)
    with torch.no_grad():
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(2):
                m.forward_mixed(x, dl, dom_dev)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        n0 = lib.mdv_launch_count()
        with torch.cuda.graph(graph):
            out = m.forward_mixed(x, dl, dom_dev)
        n_mixed = lib.mdv_launch_count() - n0
        dom_dev.copy_(torch.tensor(doms_b, dtype=torch.int32))
        graph.replay()
        torch.cuda.synchronize(dev)
        want = m.forward_mixed(x, dl, doms_b)
        assert torch.equal(out, want) or rel(out, want) <= 1e-5
        n0 = lib.mdv_launch_count()
        _main(m, x, dl, "1")
        assert lib.mdv_launch_count() - n0 == n_mixed
    del graph
