"""GPU (B200) parity tests, one per kernel family: every call goes through the C ABI (ctypes) and is compared with the
same arithmetic in plain torch fp32 (TF32 disabled) on identical seeded inputs.  Tolerances: fp32 paths 1e-4 relative to
the tensor's abs-max; paths with bf16 operands/outputs 1e-2 (bf16 has 8 mantissa bits: 2^-9 = 2e-3 per rounding)."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

BF16_TOL = 1e-2
F32_TOL = 2e-4


@pytest.fixture(scope="module")
def env():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    from mdvit_b200 import _lib as L
    return L, L.lib(), torch.device("cuda")


def rel(a, b):
    a, b = a.float(), b.float()
    return ((a - b).abs().max() / (b.abs().max() + 1e-20)).item()


# ------------------------------------------------------------------------------------------------- GEMM
@pytest.mark.parametrize("M,N,K", [(128, 64, 64), (1000, 192, 64), (300, 320, 320), (8, 512, 512), (2048, 512, 2112),
                                   (5000, 32, 64), (3000, 288, 64), (16384, 1024, 128), (777, 960, 320)])
def test_gemm_nt_shapes(env, M, N, K):
    L, lib, dev = env
    torch.manual_seed(M + N + K)
    A = torch.randn(M, K, device=dev).bfloat16()
    W = (torch.randn(N, K, device=dev) / K ** 0.5).bfloat16()
    bias = torch.randn(N, device=dev)
    res = torch.randn(M, N, device=dev)
    ref = A.float() @ W.float().t() + bias
    for out_dtype, use_res in ((torch.bfloat16, False), (torch.float32, True)):
        out = torch.empty(M, N, device=dev, dtype=out_dtype)
        e = L.GemmEpi()
        e.bias, e.out, e.ldc, e.out_bf16 = L.ptr(bias), L.ptr(out), N, int(out_dtype == torch.bfloat16)
        if use_res:
            e.residual, e.ld_res = L.ptr(res), N
        L.check(lib.mdv_gemm_nt(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(e), L.stream()), "gemm_nt")
        want = ref + res if use_res else ref
        assert rel(out, want) < (BF16_TOL if out_dtype == torch.bfloat16 else 1e-5)


@pytest.mark.parametrize("pair", [0, 1])
@pytest.mark.parametrize("M,N,K", [(256, 64, 64), (1000, 192, 64), (300, 320, 320), (2048, 512, 2112), (5000, 32, 64), (777, 960, 320),
                                   (131072, 2112, 512), (131072, 512, 2112), (524288, 192, 64)])
def test_gemm_nt_cta_pair_and_bench_sizes(env, M, N, K, pair):
    """The CTA-pair instantiation (tcgen05.mma.cta_group::2: two CTAs of a cluster share one 256-row tile) forced on and off over
    small, ragged and the benchmark's own shapes (linear_fuse forward / input gradient at B=32/domain, the stage-0 qkv GEMM at
    M = 524 288), bf16 and fp32 outputs, against torch fp32 on the same bf16 operands."""
    L, lib, dev = env
    torch.manual_seed(M + N + K)
    A = torch.randn(M, K, device=dev).bfloat16()
    W = (torch.randn(N, K, device=dev) / K ** 0.5).bfloat16()
    bias = torch.randn(N, device=dev)
    ref = torch.addmm(bias, A.float(), W.float().t())
    lib.mdv_gemm_force_pair(pair)
    try:
        for out_dtype, with_bias in ((torch.bfloat16, False), (torch.float32, True)):
            out = torch.full((M, N), float("nan"), device=dev, dtype=out_dtype)
            e = L.GemmEpi()
            e.out, e.ldc, e.out_bf16 = L.ptr(out), N, int(out_dtype == torch.bfloat16)
            if with_bias:
                e.bias = L.ptr(bias)
            L.check(lib.mdv_gemm_nt(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(e), L.stream()), "gemm_nt")
            want = ref if with_bias else ref - bias
            assert rel(out, want) < (BF16_TOL if out_dtype == torch.bfloat16 else 1e-5), (out_dtype, pair)
            del out
    finally:
        lib.mdv_gemm_force_pair(-1)


@pytest.mark.parametrize("M,N,K", [(128, 64, 64), (1000, 64, 32), (300, 320, 128), (5000, 32, 32), (3000, 64, 288), (8192, 512, 4608),
                                   (16384, 128, 64), (777, 1024, 4608), (130, 64, 36)])
def test_gemm_nt_tf32_shapes(env, M, N, K):
    """fp32 operands multiplied as TF32 (tcgen05 kind::tf32), fp32 accumulate: the conv-trunk GEMMs.  TF32 keeps 10 mantissa
    bits (2^-11 per operand rounding): 5e-4 of the output abs-max, 4x tighter than the bf16 path's 2e-3."""
    L, lib, dev = env
    torch.manual_seed(M + N + K)
    A = torch.randn(M, K, device=dev)
    W = torch.randn(N, K, device=dev) / K ** 0.5
    bias = torch.randn(N, device=dev)
    ref = A.double() @ W.double().t() + bias.double()
    for out_dtype in (torch.float32, torch.bfloat16):
        out = torch.empty(M, N, device=dev, dtype=out_dtype)
        e = L.GemmEpi()
        e.bias, e.out, e.ldc, e.out_bf16 = L.ptr(bias), L.ptr(out), N, int(out_dtype == torch.bfloat16)
        L.check(lib.mdv_gemm_nt_tf32(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(e), L.stream()), "gemm_nt_tf32")
        assert rel(out, ref.float()) < (BF16_TOL if out_dtype == torch.bfloat16 else 1e-3)
    # the same product on bf16 operands is ~4x further from the fp64 result
    out16 = torch.empty(M, N, device=dev)
    e = L.GemmEpi()
    e.bias, e.out, e.ldc, e.out_bf16 = L.ptr(bias), L.ptr(out16), N, 0
    if K % 8 == 0:
        Ab, Wb = A.bfloat16(), W.bfloat16()
        L.check(lib.mdv_gemm_nt(L.ptr(Ab), K, L.ptr(Wb), K, M, N, K, ctypes.byref(e), L.stream()), "gemm_nt")
        e32 = ((out.float() if out.dtype != torch.float32 else out) - ref.float()).norm()
        out32 = torch.empty(M, N, device=dev)
        e2 = L.GemmEpi()
        e2.bias, e2.out, e2.ldc, e2.out_bf16 = L.ptr(bias), L.ptr(out32), N, 0
        L.check(lib.mdv_gemm_nt_tf32(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(e2), L.stream()), "gemm_nt_tf32")
        assert (out32 - ref.float()).norm() < 0.5 * (out16 - ref.float()).norm()


def test_gemm_nt_gelu_preact_mulgrad_rowscale_ldc(env):
    L, lib, dev = env
    torch.manual_seed(1)
    M, N, K = 2000, 512, 128
    A = torch.randn(M, K, device=dev).bfloat16()
    W = (torch.randn(N, K, device=dev) / K ** 0.5).bfloat16()
    bias = torch.randn(N, device=dev)
    acc = A.float() @ W.float().t() + bias
    # fc1-style: pre-activation + GELU, written into a wider buffer (ldc > N)
    out = torch.zeros(M, N + 64, device=dev, dtype=torch.bfloat16)
    pre = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    e = L.GemmEpi()
    e.bias, e.out, e.ldc, e.out_bf16, e.act, e.out_preact, e.ld_preact = L.ptr(bias), L.ptr(out), N + 64, 1, L.ACT_GELU, L.ptr(pre), N
    L.check(lib.mdv_gemm_nt(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(e), L.stream()), "gemm_nt")
    assert rel(pre, acc) < BF16_TOL and rel(out[:, :N], F.gelu(acc)) < BF16_TOL
    assert out[:, N:].abs().max().item() == 0.0                    # columns beyond N untouched
    # dgrad-style: multiply by gelu'(u), per-sample row scale
    u = torch.randn(M, N, device=dev).bfloat16()
    rs = torch.rand(M // 500, device=dev) + 0.5
    out2 = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    e = L.GemmEpi()
    e.out, e.ldc, e.out_bf16, e.mul_gelu_grad, e.ld_mul, e.rowscale, e.rows_per_scale = L.ptr(out2), N, 1, L.ptr(u), N, L.ptr(rs), 500
    L.check(lib.mdv_gemm_nt(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(e), L.stream()), "gemm_nt")
    uf = u.float().requires_grad_()
    F.gelu(uf).sum().backward()
    want = (acc - bias) * uf.grad * rs.repeat_interleave(500)[:, None]
    assert rel(out2, want) < BF16_TOL
    # preact_mode 1: the forward stores gelu'(v) * dropout scale itself, the backward multiplies by it (mul_mode 1)
    rng = torch.tensor([5, 9], dtype=torch.int64, device=dev)
    fac = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    out3 = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    e = L.GemmEpi()
    e.bias, e.out, e.ldc, e.out_bf16, e.act, e.out_preact, e.ld_preact, e.preact_mode = L.ptr(bias), L.ptr(out3), N, 1, L.ACT_GELU, L.ptr(fac), N, 1
    e.dropout_p, e.rng, e.drop_stream = 0.25, L.ptr(rng), 4
    L.check(lib.mdv_gemm_nt(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(e), L.stream()), "gemm_nt")
    mask = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    L.check(lib.mdv_cast_bf16(L.ptr(torch.ones(M, N, device=dev)), N, L.ptr(mask), N, M, N, None, 1, 0.25, L.ptr(rng), 4, None, L.stream()), "cast")
    keep = (mask.float() != 0).float() / 0.75
    af = acc.clone().requires_grad_()
    F.gelu(af).sum().backward()
    assert rel(out3, F.gelu(acc) * keep) < BF16_TOL and rel(fac, af.grad * keep) < BF16_TOL
    out4 = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    e = L.GemmEpi()
    e.out, e.ldc, e.out_bf16, e.mul_gelu_grad, e.ld_mul, e.mul_mode = L.ptr(out4), N, 1, L.ptr(fac), N, 1
    L.check(lib.mdv_gemm_nt(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(e), L.stream()), "gemm_nt")
    assert rel(out4, (acc - bias) * fac.float()) < BF16_TOL


def test_gemm_nt_dropout_mask_is_reproducible_and_unbiased(env):
    L, lib, dev = env
    M, N, K, p = 4096, 256, 64, 0.1
    A = torch.ones(M, K, device=dev).bfloat16()
    W = torch.full((N, K), 1.0 / K, device=dev).bfloat16()
    rng = torch.tensor([123, 7], dtype=torch.int64, device=dev)
    outs = []
    for stream_id in (5, 5, 6):
        out = torch.empty(M, N, device=dev)
        e = L.GemmEpi()
        e.out, e.ldc, e.out_bf16, e.dropout_p, e.rng, e.drop_stream = L.ptr(out), N, 0, p, L.ptr(rng), stream_id
        L.check(lib.mdv_gemm_nt(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(e), L.stream()), "gemm_nt")
        outs.append(out)
    assert torch.equal(outs[0], outs[1]) and not torch.equal(outs[0], outs[2])
    vals = torch.unique(outs[0])
    assert vals.numel() == 2 and vals[0].item() == 0.0 and abs(vals[1].item() - 1 / (1 - p)) < 1e-5
    assert abs((outs[0] == 0).float().mean().item() - p) < 5e-3 and abs(outs[0].mean().item() - 1.0) < 1e-2
    # the standalone cast kernel regenerates the identical mask (used by the backward pass)
    ones = torch.ones(M, N, device=dev)
    m2 = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    L.check(lib.mdv_cast_bf16(L.ptr(ones), N, L.ptr(m2), N, M, N, None, 1, p, L.ptr(rng), 5, None, L.stream()), "cast")
    assert torch.equal(m2.float() == 0, outs[0] == 0)
    # ... and so does the cast+column-sum variant, whose sums are the bias gradient
    m3 = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    cs = torch.zeros(N, device=dev)
    L.check(lib.mdv_cast_bf16(L.ptr(ones), N, L.ptr(m3), N, M, N, None, 1, p, L.ptr(rng), 5, L.ptr(cs), L.stream()), "cast")
    assert torch.equal(m3, m2) and rel(cs, m2.float().sum(0)) < 1e-2


@pytest.mark.parametrize("M,N,K", [(1000, 192, 64), (5000, 512, 64), (300, 320, 1280), (40000, 1024, 128)])
def test_gemm_nt_colsum_byproduct(env, M, N, K):
    """epi.colsum accumulates the column sums of the stored tile (bias gradient of the producing Linear)."""
    L, lib, dev = env
    torch.manual_seed(N)
    A = torch.randn(M, K, device=dev).bfloat16()
    W = (torch.randn(N, K, device=dev) / K ** 0.5).bfloat16()
    for dt in (torch.bfloat16, torch.float32):
        out = torch.empty(M, N, device=dev, dtype=dt)
        cs = torch.ones(N, device=dev)
        e = L.GemmEpi()
        e.out, e.ldc, e.out_bf16, e.colsum = L.ptr(out), N, int(dt == torch.bfloat16), L.ptr(cs)
        L.check(lib.mdv_gemm_nt(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(e), L.stream()), "gemm_nt")
        ref = A.float() @ W.float().t()
        assert rel(out, ref) < BF16_TOL
        want = 1.0 + out.double().sum(0)
        assert ((cs.double() - want).abs().max() / want.abs().max()).item() < 1e-4


@pytest.mark.parametrize("M,C", [(1000, 64), (777, 128), (500, 320), (300, 512)])
def test_layernorm_bwd_masked_output_and_bias_colsum(env, M, C):
    L, lib, dev = env
    torch.manual_seed(C + 1)
    x, dy, dres = torch.randn(M, C, device=dev), torch.randn(M, C, device=dev), torch.randn(M, C, device=dev)
    g, b = 1 + 0.1 * torch.randn(C, device=dev), torch.zeros(C, device=dev)
    y = torch.empty(M, C, device=dev, dtype=torch.bfloat16)
    mean, rstd = torch.empty(M, device=dev), torch.empty(M, device=dev)
    L.check(lib.mdv_layernorm_fwd(L.ptr(x), L.ptr(g), L.ptr(b), 1e-6, L.ptr(y), L.ptr(mean), L.ptr(rstd), M, C, L.stream()), "ln")
    rows_per = 100
    rs = torch.rand((M + rows_per - 1) // rows_per, device=dev) + 0.5
    rng = torch.tensor([9, 3], dtype=torch.int64, device=dev)
    dx, dxm = torch.empty(M, C, device=dev), torch.empty(M, C, device=dev, dtype=torch.bfloat16)
    dg, db, dbm = torch.zeros(C, device=dev), torch.zeros(C, device=dev), torch.zeros(C, device=dev)
    L.check(lib.mdv_layernorm_bwd(L.ptr(dy), L.ptr(x), L.ptr(mean), L.ptr(rstd), L.ptr(g), L.ptr(dres), L.ptr(dx), L.ptr(dxm), L.ptr(rs),
                                  rows_per, 0.1, L.ptr(rng), 11, L.ptr(dg), L.ptr(db), L.ptr(dbm), M, C, L.stream()), "ln_bwd")
    mask = torch.empty(M, C, device=dev, dtype=torch.bfloat16)      # the same mask from the standalone cast kernel
    L.check(lib.mdv_cast_bf16(L.ptr(torch.ones(M, C, device=dev)), C, L.ptr(mask), C, M, C, None, 1, 0.1, L.ptr(rng), 11, None, L.stream()), "cast")
    want = dx * rs.repeat_interleave(rows_per)[:M, None] * (mask.float() != 0) / 0.9
    assert rel(dxm, want) < BF16_TOL
    assert rel(dbm, want.sum(0)) < 1e-4


@pytest.mark.parametrize("R,P,Q", [(64, 128, 64), (1000, 64, 64), (8192, 320, 1280), (9000, 32, 64), (9000, 64, 288), (8, 512, 4608),
                                   (40000, 192, 64)])
def test_gemm_tn_accumulates(env, R, P, Q):
    L, lib, dev = env
    torch.manual_seed(R + P)
    A = torch.randn(R, P, device=dev).bfloat16()
    B = torch.randn(R, Q, device=dev).bfloat16()
    C0 = torch.randn(P, Q, device=dev)
    C = C0.clone()
    L.check(lib.mdv_gemm_tn(L.ptr(A), P, L.ptr(B), Q, R, P, Q, L.ptr(C), Q, L.stream()), "gemm_tn")
    assert rel(C, C0 + A.float().t() @ B.float()) < 1e-5


# ------------------------------------------------------------------------------------------------- norms
@pytest.mark.parametrize("M,C", [(7, 64), (1000, 128), (333, 320), (4096, 512)])
def test_layernorm_fwd_bwd(env, M, C):
    L, lib, dev = env
    torch.manual_seed(C)
    x = (torch.randn(M, C, device=dev) * 3 + 1).requires_grad_()
    g = (1 + 0.1 * torch.randn(C, device=dev)).requires_grad_()
    b = (0.1 * torch.randn(C, device=dev)).requires_grad_()
    y = torch.empty(M, C, device=dev, dtype=torch.bfloat16)
    mean, rstd = torch.empty(M, device=dev), torch.empty(M, device=dev)
    L.check(lib.mdv_layernorm_fwd(L.ptr(x), L.ptr(g), L.ptr(b), 1e-6, L.ptr(y), L.ptr(mean), L.ptr(rstd), M, C, L.stream()), "ln")
    ref = F.layer_norm(x, (C,), g, b, 1e-6)
    assert rel(y, ref) < BF16_TOL
    dy, dres = torch.randn(M, C, device=dev), torch.randn(M, C, device=dev)
    (ref * dy).sum().backward()
    dx, dg, db = torch.empty(M, C, device=dev), torch.zeros(C, device=dev), torch.zeros(C, device=dev)
    L.check(lib.mdv_layernorm_bwd(L.ptr(dy), L.ptr(x), L.ptr(mean), L.ptr(rstd), L.ptr(g), L.ptr(dres), L.ptr(dx), None, None, 1, 0.0, None,
                                  0, L.ptr(dg), L.ptr(db), None, M, C, L.stream()), "ln_bwd")
    assert rel(dx, x.grad + dres) < F32_TOL and rel(dg, g.grad) < F32_TOL and rel(db, b.grad) < F32_TOL


@pytest.mark.parametrize("M,C,act", [(512, 32, 3), (1000, 64, 3), (128, 1024, 2), (3000, 512, 2)])
def test_batchnorm_train_fwd_bwd_and_running_stats(env, M, C, act):
    L, lib, dev = env
    torch.manual_seed(C + act)
    z = (torch.randn(M, C, device=dev) * 2 + 0.5).requires_grad_()
    g = (1 + 0.1 * torch.randn(C, device=dev)).requires_grad_()
    b = (0.1 * torch.randn(C, device=dev)).requires_grad_()
    rm, rv = torch.zeros(C, device=dev), torch.ones(C, device=dev)
    rm_ref, rv_ref = rm.clone(), rv.clone()
    nbt = torch.zeros((), dtype=torch.long, device=dev)
    mean, rstd = torch.empty(C, device=dev), torch.empty(C, device=dev)
    ws = torch.empty(2 * C, dtype=torch.float64, device=dev)
    L.check(lib.mdv_bn_stats(L.ptr(z), M, C, 1e-5, 0.1, 1, L.ptr(rm), L.ptr(rv), L.ptr(nbt), L.ptr(mean), L.ptr(rstd), L.ptr(ws), L.stream()), "bn")
    y = torch.empty(M, C, device=dev)
    L.check(lib.mdv_bn_act_fwd(L.ptr(z), L.ptr(mean), L.ptr(rstd), L.ptr(g), L.ptr(b), act, L.ptr(y), 0, M, C, L.stream()), "bn_act")
    actf = F.relu if act == 2 else F.hardswish
    ref = actf(F.batch_norm(z, rm_ref, rv_ref, g, b, True, 0.1, 1e-5))
    assert rel(y, ref) < F32_TOL and rel(rm, rm_ref) < 1e-5 and rel(rv, rv_ref) < 1e-5 and nbt.item() == 1
    dy = torch.randn(M, C, device=dev)
    (ref * dy).sum().backward()
    dz, dg, db = torch.empty(M, C, device=dev), torch.zeros(C, device=dev), torch.zeros(C, device=dev)
    ws2 = torch.empty(3 * C, dtype=torch.float64, device=dev)
    L.check(lib.mdv_bn_act_bwd(L.ptr(dy), L.ptr(z), L.ptr(mean), L.ptr(rstd), L.ptr(g), L.ptr(b), act, L.ptr(dz), 0, L.ptr(dg), L.ptr(db), M, C,
                               L.ptr(ws2), L.stream()), "bn_bwd")
    assert rel(dz, z.grad) < 1e-3 and rel(dg, g.grad) < 1e-3 and rel(db, b.grad) < 1e-3
    # eval mode uses the running buffers
    L.check(lib.mdv_bn_stats(None, M, C, 1e-5, 0.1, 0, L.ptr(rm), L.ptr(rv), None, L.ptr(mean), L.ptr(rstd), None, L.stream()), "bn_eval")
    assert rel(mean, rm) == 0 and rel(rstd, torch.rsqrt(rv + 1e-5)) < 1e-6


@pytest.mark.parametrize("G,Mg,C,act,bf16_out", [(4, 512, 32, 3, False), (4, 1000, 64, 3, True), (1, 128, 1024, 2, False), (4, 3000, 320, 2, False),
                                                  (2, 4096, 512, 2, True), (4, 77, 128, 3, False)])
def test_batchnorm_shared_set_table_equals_consecutive_batchnorm_calls(env, G, Mg, C, act, bf16_out):
    """mdv_bn_train_fwd_gp / mdv_bn_act_bwd_gp on G stacked mini-batches with tables that repeat one parameter set G times ==
    G consecutive nn.BatchNorm2d forwards (train mode: per-group batch statistics, running buffers updated in group order,
    num_batches_tracked += G) and their autograd (gradients summed over the groups)."""
    L, lib, dev = env
    torch.manual_seed(G * C + Mg)
    M = G * Mg
    z = (torch.randn(M, C, device=dev) * 2 + torch.arange(G, device=dev).repeat_interleave(Mg)[:, None] * 0.7).requires_grad_()
    g = (1 + 0.1 * torch.randn(C, device=dev)).requires_grad_()
    b = (0.1 * torch.randn(C, device=dev)).requires_grad_()
    rm, rv = torch.randn(C, device=dev) * 0.1, 1 + 0.2 * torch.rand(C, device=dev)
    rm_ref, rv_ref = rm.clone(), rv.clone()
    nbt = torch.zeros((), dtype=torch.long, device=dev)
    mean, rstd = torch.empty(G, C, device=dev), torch.empty(G, C, device=dev)
    y = torch.empty(M, C, device=dev, dtype=torch.bfloat16 if bf16_out else torch.float32)
    ws = torch.empty(2 * C * G, dtype=torch.float64, device=dev)
    L.check(lib.mdv_bn_train_fwd_gp(L.ptr(z), G, Mg, C, 1e-5, 0.1, L.ptr_table([rm] * G), L.ptr_table([rv] * G), L.ptr_table([nbt] * G),
                                    L.ptr_table([g] * G), L.ptr_table([b] * G), act, L.ptr(mean), L.ptr(rstd), L.ptr(y), int(bf16_out), L.ptr(ws),
                                    L.stream()), "bn_g")
    actf = F.relu if act == 2 else F.hardswish
    ref = torch.cat([actf(F.batch_norm(z[i * Mg:(i + 1) * Mg], rm_ref, rv_ref, g, b, True, 0.1, 1e-5)) for i in range(G)])
    assert rel(y, ref) < (BF16_TOL if bf16_out else F32_TOL)
    assert rel(rm, rm_ref) < 1e-5 and rel(rv, rv_ref) < 1e-5 and nbt.item() == G
    dy = torch.randn(M, C, device=dev)
    (ref * dy).sum().backward()
    dz, dg, db = torch.empty(M, C, device=dev), torch.zeros(C, device=dev), torch.zeros(C, device=dev)
    ws2 = torch.empty(3 * C * G, dtype=torch.float64, device=dev)
    L.check(lib.mdv_bn_act_bwd_gp(L.ptr(dy), L.ptr(z), L.ptr(mean), L.ptr(rstd), L.ptr_table([g] * G), L.ptr_table([b] * G), act, L.ptr(dz), 0,
                                  L.ptr_table([dg] * G), L.ptr_table([db] * G), G, Mg, C, L.ptr(ws2), L.stream()), "bn_bwd_g")
    assert rel(dz, z.grad) < 1e-3 and rel(dg, g.grad) < 1e-3 and rel(db, b.grad) < 1e-3


# ------------------------------------------------------------------------------------------------- stencils
@pytest.mark.parametrize("B,H,W,C,stride", [(2, 16, 16, 64, 1), (2, 16, 16, 64, 2), (1, 8, 12, 320, 2), (3, 4, 4, 512, 1),
                                            (2, 64, 64, 64, 1), (1, 24, 40, 128, 1), (2, 16, 20, 320, 1), (1, 70, 9, 64, 1)])
def test_dwconv3_fwd_transposed_wgrad(env, B, H, W, C, stride):
    L, lib, dev = env
    torch.manual_seed(C + stride)
    x = torch.randn(B, H, W, C, device=dev).requires_grad_()
    w = (torch.randn(C, 1, 3, 3, device=dev) * 0.3).requires_grad_()
    bias = torch.randn(C, device=dev).requires_grad_()
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    ref = F.conv2d(x.permute(0, 3, 1, 2), w, bias, stride=stride, padding=1, groups=C).permute(0, 2, 3, 1)
    out = torch.empty(B, Ho, Wo, C, device=dev)
    L.check(lib.mdv_dwconv3(L.ptr(x), L.ptr(w), L.ptr(bias), L.ptr(out), 0, B, H, W, Ho, Wo, C, stride, 0, 0, L.stream()), "dwconv")
    assert rel(out, ref) < F32_TOL
    dy = torch.randn(B, Ho, Wo, C, device=dev)
    (ref * dy).sum().backward()
    dx = torch.empty(B, H, W, C, device=dev)
    L.check(lib.mdv_dwconv3(L.ptr(dy), L.ptr(w), None, L.ptr(dx), 0, B, Ho, Wo, H, W, C, stride, 1, 0, L.stream()), "dwconv_t")
    dw, db = torch.zeros_like(w), torch.zeros_like(bias)
    L.check(lib.mdv_dwconv3_wgrad(L.ptr(dy), L.ptr(x), L.ptr(dw), L.ptr(db), B, H, W, Ho, Wo, C, stride, L.stream()), "dwconv_w")
    assert rel(dx, x.grad) < F32_TOL and rel(dw, w.grad) < F32_TOL and rel(db, bias.grad) < F32_TOL
    if stride == 1:      # ConvPosEnc form (mpvit.py:239-248): + identity, and the bf16-output variant
        out2 = torch.empty(B, H, W, C, device=dev)
        L.check(lib.mdv_dwconv3(L.ptr(x), L.ptr(w), L.ptr(bias), L.ptr(out2), 0, B, H, W, H, W, C, 1, 0, 1, L.stream()), "dwconv_res")
        assert rel(out2, ref + x) < F32_TOL
        out3 = torch.empty(B, H, W, C, device=dev, dtype=torch.bfloat16)
        L.check(lib.mdv_dwconv3(L.ptr(x), L.ptr(w), None, L.ptr(out3), 1, B, H, W, H, W, C, 1, 0, 0, L.stream()), "dwconv_bf16")
        assert rel(out3, ref - bias) < BF16_TOL
        dx2 = torch.empty(B, H, W, C, device=dev)
        L.check(lib.mdv_dwconv3(L.ptr(dy), L.ptr(w), None, L.ptr(dx2), 0, B, H, W, H, W, C, 1, 1, 1, L.stream()), "dwconv_t_res")
        assert rel(dx2, x.grad + dy) < F32_TOL


@pytest.mark.parametrize("B,H,W,C", [(2, 8, 8, 128), (2, 64, 64, 64), (1, 20, 12, 320), (3, 5, 7, 512), (1, 33, 16, 64)])
def test_gconv2_matches_grouped_conv_over_concat(env, B, H, W, C):
    L, lib, dev = env
    torch.manual_seed(3)
    skip = torch.randn(B, H, W, C, device=dev).requires_grad_()
    up = torch.randn(B, H, W, C, device=dev).requires_grad_()
    w = (torch.randn(C, 2, 3, 3, device=dev) * 0.3).requires_grad_()
    cat = torch.cat((skip, up), dim=3).permute(0, 3, 1, 2)
    ref = F.conv2d(cat, w, None, padding=1, groups=C).permute(0, 2, 3, 1)          # Decoders.py:30-38
    out = torch.empty(B, H, W, C, device=dev, dtype=torch.bfloat16)
    L.check(lib.mdv_gconv2_fwd(L.ptr(skip), L.ptr(up), L.ptr(w), L.ptr(out), 1, B, H, W, C, L.stream()), "gconv2")
    assert rel(out, ref) < BF16_TOL
    out32 = torch.empty(B, H, W, C, device=dev)                                   # fp32 output: the TF32 pointwise conv's operand
    L.check(lib.mdv_gconv2_fwd(L.ptr(skip), L.ptr(up), L.ptr(w), L.ptr(out32), 0, B, H, W, C, L.stream()), "gconv2")
    assert rel(out32, ref) < F32_TOL
    dy = torch.randn(B, H, W, C, device=dev)
    (ref * dy).sum().backward()
    ds, du, dw = torch.empty_like(skip), torch.empty_like(up), torch.zeros_like(w)
    L.check(lib.mdv_gconv2_bwd(L.ptr(dy), L.ptr(skip), L.ptr(up), L.ptr(w), L.ptr(ds), L.ptr(du), L.ptr(dw), B, H, W, C, L.stream()), "gconv2_b")
    assert rel(ds, skip.grad) < F32_TOL and rel(du, up.grad) < F32_TOL and rel(dw, w.grad) < F32_TOL


@pytest.mark.parametrize("stride,C", [(1, 64), (2, 32)])
def test_im2col_col2im_are_transposes_of_conv3x3(env, stride, C):
    L, lib, dev = env
    torch.manual_seed(stride)
    B, H, W, Cout = 2, 8, 8, 64
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    x = torch.randn(B, H, W, C, device=dev).bfloat16().float().requires_grad_()
    w = (torch.randn(Cout, C, 3, 3, device=dev) / (9 * C) ** 0.5).bfloat16().float()
    ref = F.conv2d(x.permute(0, 3, 1, 2), w, None, stride=stride, padding=1).permute(0, 2, 3, 1)
    col = torch.empty(B * Ho * Wo, 9 * C, device=dev, dtype=torch.bfloat16)
    L.check(lib.mdv_im2col3(L.ptr(x), 0, L.ptr(col), 1, B, H, W, Ho, Wo, C, stride, 9 * C, L.stream()), "im2col")
    wp = torch.zeros(Cout, 9 * C, device=dev, dtype=torch.bfloat16)
    L.check(lib.mdv_prep_weight(L.ptr(w), L.ptr(wp), Cout, 9 * C, 9 * C, 2, C, L.stream()), "prep")
    assert rel(col.float() @ wp.float().t(), ref.reshape(-1, Cout)) < 1e-4
    # fp32 variants (operands of the TF32 GEMM): identical values, fp32 storage; and the GEMM itself against F.conv2d
    col32 = torch.empty(B * Ho * Wo, 9 * C, device=dev)
    L.check(lib.mdv_im2col3(L.ptr(x), 0, L.ptr(col32), 0, B, H, W, Ho, Wo, C, stride, 9 * C, L.stream()), "im2col")
    wp32 = torch.zeros(Cout, 9 * C, device=dev)
    L.check(lib.mdv_prep_weight(L.ptr(w), L.ptr(wp32), Cout, 9 * C, 9 * C, 2 | 8, C, L.stream()), "prep")
    assert torch.equal(col32, col.float()) and torch.equal(wp32, wp.float())
    out = torch.empty(B * Ho * Wo, Cout, device=dev)
    e = L.GemmEpi()
    e.out, e.ldc, e.out_bf16 = L.ptr(out), Cout, 0
    L.check(lib.mdv_gemm_nt_tf32(L.ptr(col32), 9 * C, L.ptr(wp32), 9 * C, B * Ho * Wo, Cout, 9 * C, ctypes.byref(e), L.stream()), "gemm_tf32")
    assert rel(out, ref.reshape(-1, Cout)) < 1e-4
    dcol = torch.randn(B * Ho * Wo, 9 * C, device=dev)
    colr = F.unfold(x.permute(0, 3, 1, 2), 3, padding=1, stride=stride)            # [B, C*9, L] with (c, tap) ordering
    colr = colr.reshape(B, C, 9, Ho * Wo).permute(0, 3, 2, 1).reshape(B * Ho * Wo, 9 * C)
    assert rel(col, colr) < 1e-6
    (colr * dcol).sum().backward()
    dx = torch.empty(B, H, W, C, device=dev)
    L.check(lib.mdv_col2im3(L.ptr(dcol), L.ptr(dx), B, H, W, Ho, Wo, C, stride, 9 * C, L.stream()), "col2im")
    assert rel(dx, x.grad) < F32_TOL


@pytest.mark.parametrize("hi,ho,C", [(8, 16, 64), (4, 16, 512), (2, 16, 64), (16, 64, 1), (5, 13, 8), (8, 64, 64), (3, 40, 16), (64, 256, 1),
                                     (7, 64, 4)])
def test_bilinear_resize_and_transpose(env, hi, ho, C):
    L, lib, dev = env
    torch.manual_seed(hi * ho)
    B = 2
    x = torch.randn(B, hi, hi, C, device=dev).requires_grad_()
    ref = F.interpolate(x.permute(0, 3, 1, 2), size=(ho, ho), mode="bilinear", align_corners=False).permute(0, 2, 3, 1)
    out = torch.empty(B, ho, ho, C, device=dev)
    L.check(lib.mdv_upsample_fwd(L.ptr(x), 0, C, L.ptr(out), 0, C, B, hi, hi, ho, ho, C, L.stream()), "up")
    assert rel(out, ref) < 1e-5
    dy = torch.randn(B, ho, ho, C, device=dev)
    (ref * dy).sum().backward()
    dx = torch.empty(B, hi, hi, C, device=dev)
    L.check(lib.mdv_upsample_bwd(L.ptr(dy), 0, C, L.ptr(dx), C, B, hi, hi, ho, ho, C, None, L.stream()), "up_b")
    if C % 4 == 0 and ho % hi == 0 and ho // hi in (4, 8):        # separable two-pass form: same result
        dx2, ws = torch.empty_like(dx), torch.empty(B * ho * hi * C, device=dev)
        L.check(lib.mdv_upsample_bwd(L.ptr(dy), 0, C, L.ptr(dx2), C, B, hi, hi, ho, ho, C, L.ptr(ws), L.stream()), "up_b2")
        assert rel(dx2, dx) < 1e-5
    assert rel(dx, x.grad) < 1e-5


# ------------------------------------------------------------------------------------------------- heads / losses / optimizer
def test_rowdot_with_dropout2d_fwd_bwd(env):
    L, lib, dev = env
    torch.manual_seed(11)
    B, N, C, p = 3, 64, 512, 0.25
    x = torch.randn(B * N, C, device=dev)
    w, bias = torch.randn(C, device=dev), torch.randn(1, device=dev)
    rng = torch.tensor([9, 2], dtype=torch.int64, device=dev)
    ones = torch.ones(B * N, C, device=dev)
    mask = torch.empty(B * N, device=dev)      # recover the (sample, channel) mask by probing with unit vectors
    out = torch.empty(B * N, device=dev)
    L.check(lib.mdv_rowdot_fwd(L.ptr(x), 0, L.ptr(w), L.ptr(bias), L.ptr(out), B * N, C, N, p, L.ptr(rng), 3, L.stream()), "rowdot")
    dlog = torch.randn(B * N, device=dev)
    dx, dw, db = torch.empty(B * N, C, device=dev), torch.zeros(C, device=dev), torch.zeros(1, device=dev)
    L.check(lib.mdv_rowdot_bwd(L.ptr(dlog), L.ptr(x), 0, L.ptr(w), L.ptr(dx), L.ptr(dw), L.ptr(db), B * N, C, N, p, L.ptr(rng), 3, L.stream()), "rowdot_b")
    m = dx / (dlog[:, None] * w[None, :])                       # = mask(b, c) / (1 - p)
    mb = m.reshape(B, N, C)
    assert (mb - mb[:, :1]).abs().max().item() < 1e-4            # whole (sample, channel) planes share one draw (Dropout2d)
    keep = (mb[:, 0] > 0.5).float()
    assert abs(keep.mean().item() - (1 - p)) < 0.06
    meff = (keep / (1 - p)).repeat_interleave(N, dim=0)
    assert rel(out, (x * meff * w).sum(1) + bias) < 1e-4
    assert rel(dw, (dlog[:, None] * x * meff).sum(0)) < 1e-4 and rel(db, dlog.sum().reshape(1)) < 1e-4
    del ones, mask


@pytest.mark.parametrize("p", [0.0, 0.1])
def test_bn_backward_with_rank1_output_gradient(env, p):
    """mdv_bn_act_bwd_rank1 (dy generated on the fly from dlog, w_out and the Dropout2d mask) == mdv_bn_act_bwd on the
    dense dy that mdv_rowdot_bwd materialises."""
    L, lib, dev = env
    torch.manual_seed(11)
    B, HW, C = 3, 200, 64
    M = B * HW
    z = torch.randn(M, C, device=dev) * 2 + 0.5
    gam, bet = 1 + 0.1 * torch.randn(C, device=dev), 0.1 * torch.randn(C, device=dev)
    mean, var = z.mean(0), z.var(0, unbiased=False)
    rstd = (var + 1e-5).rsqrt()
    a5 = torch.relu((z - mean) * rstd * gam + bet).bfloat16()
    dlog, w = torch.randn(M, device=dev), torch.randn(C, device=dev)
    rng = torch.tensor([3, 1], dtype=torch.int64, device=dev)
    dense = torch.empty(M, C, device=dev)
    dw, db = torch.zeros(C, device=dev), torch.zeros(1, device=dev)
    L.check(lib.mdv_rowdot_bwd(L.ptr(dlog), L.ptr(a5), 1, L.ptr(w), L.ptr(dense), L.ptr(dw), L.ptr(db), M, C, HW, p, L.ptr(rng), 9, L.stream()), "rowdot_bwd")
    outs = []
    for rank1 in (False, True):
        dz = torch.empty(M, C, device=dev)
        dg, dbt = torch.zeros(C, device=dev), torch.zeros(C, device=dev)
        ws = torch.empty(3 * C + (B * C + 1) // 2, dtype=torch.float64, device=dev)      # + the [samples, C] factor table of the rank-1 form
        if rank1:
            L.check(lib.mdv_bn_act_bwd_rank1(L.ptr(dlog), L.ptr(w), HW, p, L.ptr(rng), 9, L.ptr(z), L.ptr(mean), L.ptr(rstd), L.ptr(gam), L.ptr(bet), 2,
                                             L.ptr(dz), 0, L.ptr(dg), L.ptr(dbt), M, C, L.ptr(ws), L.stream()), "bn_bwd_rank1")
        else:
            L.check(lib.mdv_bn_act_bwd(L.ptr(dense), L.ptr(z), L.ptr(mean), L.ptr(rstd), L.ptr(gam), L.ptr(bet), 2, L.ptr(dz), 0, L.ptr(dg), L.ptr(dbt),
                                       M, C, L.ptr(ws), L.stream()), "bn_bwd")
        outs.append((dz, dg, dbt))
    for a, b in zip(outs[0], outs[1]):
        assert rel(b, a) < 1e-5
    # dx == NULL: weight gradients only
    dw2, db2 = torch.zeros(C, device=dev), torch.zeros(1, device=dev)
    L.check(lib.mdv_rowdot_bwd(L.ptr(dlog), L.ptr(a5), 1, L.ptr(w), None, L.ptr(dw2), L.ptr(db2), M, C, HW, p, L.ptr(rng), 9, L.stream()), "rowdot_bwd")
    assert rel(dw2, dw) < 1e-5 and rel(db2, db) < 1e-5


def test_fused_losses_match_reference_formulas(env):
    L, lib, dev = env
    from oracle import mdvit_oracle as O
    torch.manual_seed(5)
    n = 2 * 64 * 64
    out = (torch.randn(n, device=dev) * 3).requires_grad_()
    aux = (torch.randn(n, device=dev) * 3).requires_grad_()
    out.data[:4] = torch.tensor([120.0, -120.0, 40.0, -40.0], device=dev)     # saturated sigmoids: BCE log clamp at -100
    y = (torch.rand(n, device=dev) < 0.3).float()
    sums = torch.empty(8, dtype=torch.float64, device=dev)
    losses = torch.empty(3, device=dev)
    L.check(lib.mdv_loss_sums(L.ptr(out), L.ptr(aux), L.ptr(y), 0, L.ptr(sums), n, L.stream()), "sums")
    L.check(lib.mdv_loss_finalize(L.ptr(sums), float(n), L.ptr(losses), L.stream()), "fin")
    ref = O.seg_losses(out, aux, y)
    for a, b in zip(losses, ref):
        assert abs(a.item() - b.item()) < 2e-5 * max(1.0, abs(b.item()))
    # uint8 labels (a quarter of the host->device bytes): identical sums
    sums8 = torch.empty(8, dtype=torch.float64, device=dev)
    y8 = y.to(torch.uint8)
    L.check(lib.mdv_loss_sums(L.ptr(out), L.ptr(aux), L.ptr(y8), 1, L.ptr(sums8), n, L.stream()), "sums8")
    assert (sums8 - sums).abs().max().item() <= 1e-9 * sums.abs().max().item()
    coef = torch.tensor([0.5, 1.0, 0.5], device=dev)
    # gradient reference: nn.BCELoss's own backward (the oracle's log().clamp() formula gives 0*inf = nan at saturated
    # sigmoids, where PyTorch's BCELoss backward — and the reference trainer — give 0)
    p, q = torch.sigmoid(out), torch.sigmoid(aux)
    bce = torch.nn.BCELoss()
    l_seg, l_aux, l_kt = bce(p, y) + O.dice_loss(p, y), bce(q, y) + O.dice_loss(q, y), O.dice_loss(q, p)
    (0.5 * l_seg + l_aux + 0.5 * l_kt).backward()
    dout, daux = torch.empty(n, device=dev), torch.empty(n, device=dev)
    L.check(lib.mdv_loss_bwd(L.ptr(out), L.ptr(aux), L.ptr(y), 0, L.ptr(sums), float(n), L.ptr(coef), L.ptr(dout), L.ptr(daux), n, L.stream()), "lb")
    assert rel(dout, out.grad) < 1e-4 and rel(daux, aux.grad) < 1e-4
    dout8, daux8 = torch.empty(n, device=dev), torch.empty(n, device=dev)
    L.check(lib.mdv_loss_bwd(L.ptr(out), L.ptr(aux), L.ptr(y8), 1, L.ptr(sums), float(n), L.ptr(coef), L.ptr(dout8), L.ptr(daux8), n, L.stream()), "lb8")
    assert torch.equal(dout8, dout) and torch.equal(daux8, daux)


def test_adamw_matches_torch(env):
    L, lib, dev = env
    torch.manual_seed(2)
    n = 100003
    p = torch.randn(n + 1, device=dev)[:n]
    p = torch.randn(n, device=dev)
    g = torch.randn(n, device=dev) * 0.01
    ref = p.clone().requires_grad_()
    opt = torch.optim.AdamW([ref], lr=1e-4, weight_decay=0.05)
    m, v = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    # the step count t lives in hyper[5] on the device and is bumped by the call itself (graph replays need no host input)
    hyper = torch.tensor([1e-4, 0.9, 0.999, 1e-8, 0.05, 0.0, 0.0, 1.0], dtype=torch.float64, device=dev)
    for t in range(1, 8):
        ref.grad = g * t
        opt.step()
        gt = (g * t).contiguous()
        L.check(lib.mdv_adamw(L.ptr(p), L.ptr(gt), L.ptr(m), L.ptr(v), L.ptr(hyper), n, L.stream()), "adamw")
    assert int(hyper[5].item()) == 7
    assert (p - ref.detach()).abs().max().item() < 5e-7      # 2 ulp at |p| ~ 2


def test_da_gate_fwd_bwd(env):
    L, lib, dev = env
    from oracle import mdvit_oracle as O
    torch.manual_seed(4)
    B, C, hid, nd = 5, 128, 64, 4
    sd = {"a.domain_layer.0.weight": torch.randn(hid, nd, device=dev).requires_grad_(), "a.domain_layer.0.bias": torch.randn(hid, device=dev).requires_grad_(),
          "a.domain_layer.2.weight": (torch.randn(C, hid, device=dev) * 0.3).requires_grad_(), "a.domain_layer.2.bias": torch.randn(C, device=dev).requires_grad_()}
    label = F.one_hot(torch.tensor([0, 3, 1, 2, 3]), nd).float().to(dev)
    ref = O.domain_gate(sd, "a", label, 8).reshape(B, C)
    gate, hidb = torch.empty(B, C, device=dev), torch.empty(B, hid, device=dev)
    P = [L.ptr(sd[k]) for k in sd]
    L.check(lib.mdv_da_gate_fwd(L.ptr(label), P[0], P[1], P[2], P[3], L.ptr(hidb), L.ptr(gate), B, nd, hid, C, 8, L.stream()), "da")
    assert rel(gate, ref) < 1e-5
    dgate = torch.randn(B, C, device=dev)
    (ref * dgate).sum().backward()
    gr = [torch.zeros_like(sd[k]) for k in sd]
    ws = torch.empty(B * (C + hid), device=dev)
    L.check(lib.mdv_da_gate_bwd(L.ptr(label), P[2], L.ptr(hidb), L.ptr(gate), L.ptr(dgate), L.ptr(gr[0]), L.ptr(gr[1]), L.ptr(gr[2]), L.ptr(gr[3]),
                                L.ptr(ws), B, nd, hid, C, 8, L.stream()), "da_b")
    for gmine, k in zip(gr, sd):
        assert rel(gmine, sd[k].grad) < 1e-4, k


# ------------------------------------------------------------------------------------------------- attention
@pytest.mark.parametrize("B,H,W,C,sup", [(2, 16, 16, 64, True), (2, 8, 8, 128, True), (2, 4, 4, 320, True), (2, 2, 2, 512, True),
                                         (3, 12, 20, 64, True), (1, 40, 24, 128, False), (2, 16, 16, 320, True), (2, 8, 8, 512, False),
                                         (2, 64, 64, 64, True), (1, 32, 32, 128, True), (1, 20, 36, 320, True), (1, 17, 9, 512, True)])
def test_factorized_attention_fwd_bwd(env, B, H, W, C, sup):
    L, lib, dev = env
    from oracle import mdvit_oracle as O
    torch.manual_seed(C + H)
    Ch, N, P = C // 8, H * W, L.ptr
    qkv = torch.randn(B, N, 3 * C, device=dev).bfloat16()
    sd = {}
    for i, (win, hh) in enumerate(((3, 2), (5, 3), (7, 3))):
        sd[f"crpe.conv_list.{i}.weight"] = (torch.randn(hh * Ch, 1, win, win, device=dev) * 0.2).requires_grad_()
        sd[f"crpe.conv_list.{i}.bias"] = (torch.randn(hh * Ch, device=dev) * 0.2).requires_grad_()
    gate = torch.softmax(torch.randn(B, 8, Ch, device=dev), dim=1).reshape(B, C).contiguous() if sup else None
    q32 = qkv.float().requires_grad_()
    t = q32.reshape(B, N, 3, 8, Ch).permute(2, 0, 3, 1, 4)
    q, k, v = t[0], t[1], t[2]
    fa = (Ch ** -0.5) * torch.einsum("bhnk,bhkv->bhnv", q, torch.einsum("bhnk,bhnv->bhkv", k.softmax(dim=2), v)) \
        + O.conv_rel_pos_enc(sd, "crpe", q, v, H, W)                                  # mdvit.py:293-298
    gref = gate.clone().requires_grad_() if sup else None
    if sup:
        fa = gref.reshape(B, 8, 1, Ch) * fa                                           # mdvit.py:304
    yref = fa.transpose(1, 2).reshape(B, N, C)
    stats = torch.empty(lib.mdv_attn_stats_floats(B, C, 8), device=dev)
    ws = torch.empty(lib.mdv_attn_ws_floats(B, C, 8), device=dev)
    y = torch.empty(B, N, C, device=dev, dtype=torch.bfloat16)
    cw = [sd[f"crpe.conv_list.{i}.{n}"].detach() for i in range(3) for n in ("weight", "bias")]
    ecrpe = torch.empty(B, N, C, device=dev, dtype=torch.bfloat16)
    L.check(lib.mdv_attn_fwd(P(qkv), P(gate), *[P(t_) for t_ in cw], P(stats), P(ws), P(y), P(ecrpe), B, H, W, C, 8, L.stream()), "attn_fwd")
    assert rel(y, yref) < BF16_TOL
    y2 = torch.empty_like(y)                       # no atomics in the forward: bit-reproducible
    L.check(lib.mdv_attn_fwd(P(qkv), P(gate), *[P(t_) for t_ in cw], P(stats), P(ws), P(y2), None, B, H, W, C, 8, L.stream()), "attn_fwd")
    assert torch.equal(y, y2)
    dy = torch.randn(B, N, C, device=dev).bfloat16()
    yref.backward(dy.float())
    dqkv = torch.empty_like(qkv)
    dgate = torch.full((B, C), float("nan"), device=dev) if sup else None      # overwritten by the call
    gcw = [torch.zeros_like(t_) for t_ in cw]
    dbq = torch.zeros(3 * C, device=dev)
    L.check(lib.mdv_attn_bwd(P(qkv), P(dy), P(y), P(ecrpe), P(gate), *[P(t_) for t_ in cw], P(stats), P(dqkv), P(dgate), *[P(t_) for t_ in gcw], P(dbq), P(ws),
                             B, H, W, C, 8, L.stream()), "attn_bwd")
    g = q32.grad
    for sl in (slice(0, C), slice(C, 2 * C), slice(2 * C, 3 * C)):
        assert rel(dqkv[..., sl], g[..., sl]) < BF16_TOL
    assert rel(dbq, g.sum(dim=(0, 1))) < BF16_TOL                                     # qkv bias gradient by-product
    for i in range(3):
        assert rel(gcw[2 * i], sd[f"crpe.conv_list.{i}.weight"].grad) < BF16_TOL
        assert rel(gcw[2 * i + 1], sd[f"crpe.conv_list.{i}.bias"].grad) < BF16_TOL
    if sup:
        assert rel(dgate, gref.grad) < BF16_TOL
        # activation-gradient-only mode (CRPE gradient pointers NULL): same dqkv, dgate still produced
        dqkv2, dgate2 = torch.empty_like(qkv), torch.full((B, C), float("nan"), device=dev)
        L.check(lib.mdv_attn_bwd(P(qkv), P(dy), P(y), P(ecrpe), P(gate), *[P(t_) for t_ in cw], P(stats), P(dqkv2), P(dgate2), None, None, None, None,
                                 None, None, None, P(ws), B, H, W, C, 8, L.stream()), "attn_bwd")
        assert torch.equal(dqkv2, dqkv) and rel(dgate2, gref.grad) < BF16_TOL
