"""Host-side operators of the MDViT hot path: torch.autograd.Functions whose forward/backward are sequences of
C-ABI kernel launches (include/mdvit_b200.h).  torch supplies device memory, the current stream and the autograd
tape; all arithmetic runs in libmdvit_b200.so.  Activations are token-major fp32/bf16 ([B, H*W, C] == NHWC).

Every Function tolerates being back-propagated twice over one graph (multi_train_MDViT.py:201,207 call backward
with retain_graph=True and then again): saved tensors are never written in backward, all backward scratch is
freshly allocated, and parameter gradients are returned for autograd to install (or, for a trainer that opted in, accumulated into its
own `.grad` buffers in place — see gtarget); the requires_grad flips on `domain_layer` between the two passes are
honoured at backward time.
"""
import ctypes
import itertools
import weakref

import torch

from . import _lib as L
from ._lib import ACT_GELU, ACT_HSWISH, ACT_NONE, ACT_RELU, GemmEpi, check, ptr, ptr_table

BF16, F32 = torch.bfloat16, torch.float32
HEADS = 8

# ------------------------------------------------------------------------------------------------- RNG state
_rng_state = {}
_stream_counter = itertools.count(1)


def rng_tensor(device):
    """Device uint64[2] {seed, step}: dropout masks are hash(seed, step, stream-id, element)."""
    t = _rng_state.get(device)
    if t is None:
        t = torch.tensor([0x5EED, 0], dtype=torch.int64, device=device)
        _rng_state[device] = t
    return t


def manual_seed(seed, device):
    rng_tensor(torch.device(device))[0] = int(seed)


def rng_bump(device):
    check(L.lib().mdv_rng_bump(ptr(rng_tensor(device)), L.stream()), "mdv_rng_bump")


def reset_stream_ids():
    """Call at the start of every training step so mask stream ids are reproducible (CUDA-graph friendly)."""
    global _stream_counter
    _stream_counter = itertools.count(1)


def new_stream_id():
    return next(_stream_counter) & 0xFFFFFFFF


# ------------------------------------------------------------------------------------------------- weight cache
WEIGHT_EPOCH = 0
_wcache = {}


def bump_weight_epoch():
    """Invalidate cached bf16 operand copies (called by the fused optimizer, which updates params by pointer)."""
    global WEIGHT_EPOCH
    WEIGHT_EPOCH += 1
    _wcache.clear()


class _PrepDesc(ctypes.Structure):
    _fields_ = [("src", ctypes.c_void_p), ("dst", ctypes.c_void_p), ("rows", ctypes.c_int), ("cols", ctypes.c_int), ("ld", ctypes.c_int),
                ("mode", ctypes.c_int), ("cin", ctypes.c_int), ("pad_", ctypes.c_int)]


class WeightMirror:
    """Persistent bf16 operand copies of every weight a training step uses, refreshed by ONE kernel launch.

    While `recording`, prep_weight() notes every (parameter, mode) it converts; freeze() uploads the descriptor table;
    afterwards the fused trainer calls refresh() once per step (right after AdamW) instead of ~200 tiny conversion
    launches, and prep_weight() hands out the persistent buffers."""

    def __init__(self):
        self.entries, self.table, self.recording = {}, None, True

    def note(self, w, mode, rows, cols, out_ld, cin, dst):
        if self.recording:
            self.entries[(id(w), mode, out_ld)] = (weakref.ref(w), w.data_ptr(), dst, rows, cols, out_ld, mode, cin)

    def lookup(self, w, mode, out_ld):
        if self.table is None:
            return None
        e = self.entries.get((id(w), mode, out_ld))
        if e is not None and e[0]() is w and e[1] == w.data_ptr():
            return e[2]
        return None

    def freeze(self, device):
        self.recording = False
        arr = (_PrepDesc * len(self.entries))()
        for i, (_, src, dst, rows, cols, out_ld, mode, cin) in enumerate(self.entries.values()):
            arr[i] = _PrepDesc(src, dst.data_ptr(), rows, cols, out_ld, mode, cin, 0)
        raw = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).clone()
        self.table = raw.to(device)
        self.n = len(self.entries)

    def refresh(self):
        check(L.lib().mdv_prep_weights_batched(ptr(self.table), self.n, L.stream()), "mdv_prep_weights_batched")


_mirror = None


def set_weight_mirror(m):
    global _mirror
    _mirror = m


def prep_weight(w, mode, rows, cols, ld=None, cin=0):
    """GEMM operand of fp32 parameter `w`: bf16, or fp32 (TF32 GEMM operand) when 8 is added to the mode
    (mode & 7: 0 copy [R,ld], 1 transpose [Cc,ld], 2/3 conv3x3 im2col order, 4 conv3x3 -> [Cin, tap*R + r])."""
    R, Cc = rows, cols
    m = mode & 7
    if m == 0 or m == 2:
        out_rows, out_ld = R, (ld or Cc)
    elif m == 4:      # conv3x3 [R, Cin, 3, 3] -> [Cin, 9 R] (input-gradient operand of mdv_conv3_gemm)
        out_rows, out_ld = Cc // 9, (ld or 9 * R)
    else:
        out_rows, out_ld = Cc, (ld or R)
    if _mirror is not None:
        hit = _mirror.lookup(w, mode, out_ld)
        if hit is not None:
            return hit
    key = (id(w), w.data_ptr(), w._version, mode, ld, WEIGHT_EPOCH)
    hit = _wcache.get(key)
    if hit is not None and hit[0]() is w:      # id()/data_ptr() are recycled once a model is freed: check liveness
        return hit[1]
    with torch.no_grad():
        dst = (torch.zeros if m >= 2 else torch.empty)((out_rows, out_ld), dtype=F32 if mode & 8 else BF16, device=w.device)
        check(L.lib().mdv_prep_weight(ptr(w), ptr(dst), R, Cc, out_ld, mode, cin, L.stream()), "mdv_prep_weight")
    if len(_wcache) > 4096:
        _wcache.clear()
    _wcache[key] = (weakref.ref(w), dst)
    if _mirror is not None:
        _mirror.note(w, mode, R, Cc, out_ld, cin, dst)
    return dst


# ------------------------------------------------------------------------------------------------- thin wrappers
def gemm_nt(A, W, M, N, K, out, *, lda=None, ldw=None, ldc=None, bias=None, residual=None, act=ACT_NONE, out_preact=None,
            mul_gelu_grad=None, drop_p=0.0, drop_stream=0, rowscale=None, rows_per_scale=1, accumulate=False, colsum=None,
            preact_mode=0, mul_mode=0, tf32=False, colscale=None, sample_set=None, rows_per_sample=1):
    """out = epilogue(A . W^T).  A, W bf16 — or both fp32 with tf32=True (TF32 tensor-core math: the conv trunk, see
    include/mdvit_b200.h mdv_gemm_nt_tf32).  With a sample_set (int32 [B] on the device, tf32 only), colscale / bias are [S, N]
    folded-BatchNorm tables and row m uses table row sample_set[m // rows_per_sample] (mdv_gemm_nt_tf32_sets)."""
    e = GemmEpi()
    e.bias, e.residual, e.mul_gelu_grad, e.out_preact = ptr(bias), ptr(residual), ptr(mul_gelu_grad), ptr(out_preact)
    e.out, e.rowscale, e.colsum, e.colscale = ptr(out), ptr(rowscale), ptr(colsum), ptr(colscale)
    e.rng = ptr(rng_tensor(out.device)) if drop_p > 0 else None
    e.ld_res = N if residual is not None else 0
    e.ld_mul = N if mul_gelu_grad is not None else 0
    e.ld_preact = N if out_preact is not None else 0
    e.ldc = ldc or N
    e.rows_per_scale = rows_per_scale
    e.out_bf16 = 1 if out.dtype == BF16 else 0
    e.act = act
    e.accumulate = 1 if accumulate else 0
    e.preact_mode, e.mul_mode = preact_mode, mul_mode
    e.dropout_p = float(drop_p)
    e.drop_stream = drop_stream
    if sample_set is not None:
        if not tf32 or A.dtype != F32 or W.dtype != F32:
            raise TypeError("the per-sample-set GEMM is a tf32 GEMM: it needs fp32 operands")
        check(L.lib().mdv_gemm_nt_tf32_sets(ptr(A), lda or K, ptr(W), ldw or K, M, N, K, ctypes.byref(e), ptr(sample_set), rows_per_sample,
                                            colscale.shape[0], L.stream()), "mdv_gemm_nt_tf32_sets")
    elif tf32:
        if A.dtype != F32 or W.dtype != F32:
            raise TypeError("tf32 GEMM needs fp32 operands")
        check(L.lib().mdv_gemm_nt_tf32(ptr(A), lda or K, ptr(W), ldw or K, M, N, K, ctypes.byref(e), L.stream()), "mdv_gemm_nt_tf32")
    else:
        check(L.lib().mdv_gemm_nt(ptr(A), lda or K, ptr(W), ldw or K, M, N, K, ctypes.byref(e), L.stream()), "mdv_gemm_nt")
    return out


def gemm_tn(A, B, R, P, Q, C, *, lda=None, ldb=None, ldc=None):
    """C[P,Q] += A[R,P]^T B[R,Q]   (skipped when C is None: weight gradients are off in this backward mode)"""
    if C is None:
        return None
    check(L.lib().mdv_gemm_tn(ptr(A), lda or P, ptr(B), ldb or Q, R, P, Q, ptr(C), ldc or Q, L.stream()), "mdv_gemm_tn")
    return C


def colsum(x, M, C, out, ld=None):
    if out is None:
        return None
    check(L.lib().mdv_colsum(ptr(x), int(x.dtype == BF16), ld or C, ptr(out), M, C, L.stream()), "mdv_colsum")
    return out


def cast_bf16(x, M, C, out=None, ld_in=None, ld_out=None, rowscale=None, rows_per_scale=1, drop_p=0.0, drop_stream=0, colsum=None):
    if out is None:
        out = torch.empty((M, C), dtype=BF16, device=x.device)
    check(L.lib().mdv_cast_bf16(ptr(x), ld_in or C, ptr(out), ld_out or C, M, C, ptr(rowscale), rows_per_scale, float(drop_p),
                                ptr(rng_tensor(x.device)) if drop_p > 0 else None, drop_stream, ptr(colsum), L.stream()),
          "mdv_cast_bf16")
    return out


def layernorm_fwd(x, w, b, M, C, eps=1e-6, rows_per_sample=None):
    """w, b: lists of S parameter tensors.  S = 1 normalises every row with the one set; with S > 1, rows [s M/S, (s+1) M/S)
    use set s (domain-specific norms) — or, inside norm_sets(), row m uses set sample_set[m // rows_per_sample]; mean / rstd are
    then None (inference needs neither)."""
    S = len(w)
    if S > 1 and _NORM_SETS is not None:
        if rows_per_sample is None:
            raise ValueError("per-sample norm sets need rows_per_sample")
        y = torch.empty((M, C), dtype=BF16, device=x.device)
        check(L.lib().mdv_layernorm_fwd_sets(ptr(x), ptr_table(w), ptr_table(b), ctypes.c_float(eps), ptr(y), None, None, ptr(_NORM_SETS),
                                             rows_per_sample, S, M, C, L.stream()), "mdv_layernorm_fwd_sets")
        return y, None, None
    if M % S:
        raise ValueError("LayerNorm groups must divide the batch")
    y = torch.empty((M, C), dtype=BF16, device=x.device)
    mean = torch.empty(M, dtype=F32, device=x.device)
    rstd = torch.empty(M, dtype=F32, device=x.device)
    check(L.lib().mdv_layernorm_fwd_gp(ptr(x), ptr_table(w), ptr_table(b), ctypes.c_float(eps), ptr(y), ptr(mean), ptr(rstd), S, M // S, C,
                                       L.stream()), "mdv_layernorm_fwd_gp")
    return y, mean, rstd


def layernorm_bwd(dy, x, mean, rstd, w, dres, M, C, dg, db, *, masked=False, rowscale=None, rows_per_scale=1, drop_p=0.0,
                  drop_stream=0, dbias_masked=None):
    """w, dg, db: lists of S, as in layernorm_fwd (dg / db entries may be None)."""
    S = len(w)
    dx = torch.empty((M, C), dtype=F32, device=x.device)
    dxm = torch.empty((M, C), dtype=BF16, device=x.device) if masked else None
    rng = ptr(rng_tensor(x.device)) if drop_p > 0 else None
    check(L.lib().mdv_layernorm_bwd_gp(ptr(dy), ptr(x), ptr(mean), ptr(rstd), ptr_table(w), ptr(dres), ptr(dx), ptr(dxm), ptr(rowscale),
                                       rows_per_scale, ctypes.c_float(drop_p), rng, drop_stream, ptr_table(dg), ptr_table(db),
                                       ptr(dbias_masked), S, M // S, C, L.stream()), "mdv_layernorm_bwd_gp")
    return dx, dxm


def dwconv3(x, w, bias, B, Hi, Wi, Ho, Wo, C, stride, *, out_bf16=False, transposed=False, residual=False):
    out = torch.empty((B, Ho * Wo, C), dtype=BF16 if out_bf16 else F32, device=x.device)
    check(L.lib().mdv_dwconv3(ptr(x), ptr(w), ptr(bias), ptr(out), int(out_bf16), B, Hi, Wi, Ho, Wo, C, stride, int(transposed),
                              int(residual), L.stream()), "mdv_dwconv3")
    return out


def dwconv3_wgrad(dy, x, dw, db, B, Hi, Wi, Ho, Wo, C, stride):
    if dw is None:
        return
    check(L.lib().mdv_dwconv3_wgrad(ptr(dy), ptr(x), ptr(dw), ptr(db), B, Hi, Wi, Ho, Wo, C, stride, L.stream()), "mdv_dwconv3_wgrad")


class BNState:
    """mean/rstd of one BatchNorm application (+ the buffers it updates)."""

    def __init__(self, bn, C):
        self.bn, self.C = bn, C


# BatchNorm groups: the fused multi-domain forward (model.MDViT.forward_multi) stacks the G single-domain mini-batches
# of one training step along the batch axis so that every per-sample kernel runs once on G*B samples; BatchNorm, whose
# batch statistics the reference computes per domain forward (mdvit.py:667 is called once per domain), is then
# evaluated per group of M/G consecutive rows — same kernels, on row slices; running statistics are updated group by
# group in order, exactly as G consecutive forwards would.
_BN_GROUPS = 1


class bn_groups:
    def __init__(self, g):
        self.g = int(g)

    def __enter__(self):
        global _BN_GROUPS
        self.prev, _BN_GROUPS = _BN_GROUPS, self.g

    def __exit__(self, *exc):
        global _BN_GROUPS
        _BN_GROUPS = self.prev


def current_bn_groups():
    return _BN_GROUPS


# Per-sample norm sets: the mixed-domain inference pass of the domain-specific-norm models (model.MDViT_DSN.forward_mixed) gives
# every norm Function all S sets, and sample b of the batch is normalised with set sample_set[b].  The index vector lives on the
# device and the kernels read it, so one captured graph serves any domain mix.  Eval only: the train-mode paths keep their row
# groups (bn_groups).
_NORM_SETS = None


class norm_sets:
    def __init__(self, sample_set):
        if sample_set.dtype != torch.int32 or not sample_set.is_cuda or sample_set.dim() != 1:
            raise TypeError("norm_sets takes a 1-D int32 CUDA tensor of per-sample set indices")
        self.sample_set = sample_set

    def __enter__(self):
        global _NORM_SETS
        self.prev, _NORM_SETS = _NORM_SETS, self.sample_set
        return self.sample_set

    def __exit__(self, *exc):
        global _NORM_SETS
        _NORM_SETS = self.prev


def current_norm_sets():
    return _NORM_SETS


def _check_norm_sets(training):
    if training and _NORM_SETS is not None:
        raise RuntimeError("ops.norm_sets (per-sample norm sets) is an eval-mode path; training uses per-group sets (bn_groups)")


def _one_set(*lists):
    """The tensors of a single norm parameter set: the eval-mode paths take one set (or S sets inside norm_sets)."""
    if len(lists[0]) != 1:
        raise ValueError("per-group norm sets are a train-mode path")
    return [t[0] for t in lists]


def _require_train_bn(training):
    """Backward of a Function whose forward ran BatchNorm in eval mode: that forward saved no batch statistics."""
    if not training:
        raise RuntimeError("mdvit_b200: backward through eval-mode BatchNorm is not supported")


def bn_fold(weight, bias, running_mean, running_var, conv_bias=None, eps=1e-5):
    """Eval-mode BatchNorm as (scale, shift) for the epilogue of the GEMM that feeds it (gemm_nt(colscale=scale, bias=shift,
    act=...)): the normalised tensor is produced by the GEMM itself, its fp32 pre-activation never reaches HBM.  The parameters and
    buffers are lists of S sets: S = 1 gives [C] vectors; S > 1 (inside norm_sets only) gives [S, C] tables in one launch, for
    the per-sample-set GEMM (see _conv_bn_fwd)."""
    if len(weight) > 1 and _NORM_SETS is not None:
        S, C = len(weight), weight[0].numel()
        st = torch.empty((2, S, C), dtype=F32, device=weight[0].device)
        check(L.lib().mdv_bn_fold_sets(ptr_table(weight), ptr_table(bias), ptr_table(running_mean), ptr_table(running_var), ptr(conv_bias),
                                       ctypes.c_float(eps), ptr(st[0]), ptr(st[1]), S, C, L.stream()), "mdv_bn_fold_sets")
        return st[0], st[1]
    weight, bias, running_mean, running_var = _one_set(weight, bias, running_mean, running_var)
    C = weight.numel()
    st = torch.empty((2, C), dtype=F32, device=weight.device)
    check(L.lib().mdv_bn_fold(ptr(weight), ptr(bias), ptr(running_mean), ptr(running_var), ptr(conv_bias), ctypes.c_float(eps), ptr(st[0]),
                              ptr(st[1]), C, L.stream()), "mdv_bn_fold")
    return st[0], st[1]


def bn_forward(z, M, C, weight, bias, running_mean, running_var, nbt, training, act, out_bf16, eps=1e-5, momentum=0.1):
    """weight, bias and the three buffers: lists of S parameter sets.  In training each of the G = bn_groups() row groups is
    normalised with its own batch statistics; with S = 1 the groups share the set (its buffers are updated group by group, in
    order), with S = G group g uses set g and updates only its buffers.  Eval takes S = 1."""
    dev = z.device
    z = z.view(M, C)
    y = torch.empty((M, C), dtype=BF16 if out_bf16 else F32, device=dev)
    if not training:
        weight, bias, running_mean, running_var = _one_set(weight, bias, running_mean, running_var)
        mean = torch.empty((1, C), dtype=F32, device=dev)
        rstd = torch.empty((1, C), dtype=F32, device=dev)
        check(L.lib().mdv_bn_stats(ptr(z), M, C, ctypes.c_float(eps), ctypes.c_float(momentum), 0, ptr(running_mean), ptr(running_var), None,
                                   ptr(mean), ptr(rstd), None, L.stream()), "mdv_bn_stats")
        check(L.lib().mdv_bn_act_fwd(ptr(z), ptr(mean), ptr(rstd), ptr(weight), ptr(bias), act, ptr(y), int(out_bf16), M, C, L.stream()),
              "mdv_bn_act_fwd")
        return y, mean, rstd
    G = _BN_GROUPS
    if M % G:
        raise ValueError("BatchNorm groups must divide the batch")
    if len(weight) not in (1, G):
        raise ValueError("BatchNorm takes one parameter set, or one per bn_groups() group")
    r = G // len(weight)      # table entries repeat a shared set once per group
    mean = torch.empty((G, C), dtype=F32, device=dev)
    rstd = torch.empty((G, C), dtype=F32, device=dev)
    ws = torch.empty(2 * C * G, dtype=torch.float64, device=dev)
    check(L.lib().mdv_bn_train_fwd_gp(ptr(z), G, M // G, C, ctypes.c_float(eps), ctypes.c_float(momentum), ptr_table(running_mean * r),
                                      ptr_table(running_var * r), ptr_table(nbt * r), ptr_table(weight * r), ptr_table(bias * r), act, ptr(mean),
                                      ptr(rstd), ptr(y), int(out_bf16), ptr(ws), L.stream()), "mdv_bn_train_fwd_gp")
    return y, mean, rstd


def bn_backward(dy, z, mean, rstd, weight, bias, act, M, C, dz_bf16=True):
    """Returns dz and the lists of values to return from backward for the S sets' gamma and beta (as given to bn_forward).
    mean/rstd are [G, C]: one row per group."""
    dev = z.device
    G = mean.shape[0]
    r = G // len(weight)
    dy, z = dy.view(M, C), z.view(M, C)
    dz = torch.empty((M, C), dtype=BF16 if dz_bf16 else F32, device=dev)
    ws = torch.empty(3 * C * G, dtype=torch.float64, device=dev)
    tg, tb = [gtarget(w) for w in weight], [gtarget(b) for b in bias]
    check(L.lib().mdv_bn_act_bwd_gp(ptr(dy), ptr(z), ptr(mean), ptr(rstd), ptr_table(weight * r), ptr_table(bias * r), act, ptr(dz),
                                    int(dz_bf16), ptr_table([t[0] for t in tg] * r), ptr_table([t[0] for t in tb] * r), G, M // G, C, ptr(ws),
                                    L.stream()), "mdv_bn_act_bwd_gp")
    return dz, [t[1] for t in tg], [t[1] for t in tb]


def upsample_fwd(x, out, B, Hi, Wi, Ho, Wo, C, ld_in=None, ld_out=None):
    check(L.lib().mdv_upsample_fwd(ptr(x), int(x.dtype == BF16), ld_in or C, ptr(out), int(out.dtype == BF16), ld_out or C, B, Hi, Wi,
                                   Ho, Wo, C, L.stream()), "mdv_upsample_fwd")
    return out


def upsample_bwd(dout, B, Hi, Wi, Ho, Wo, C, ld_out=None):
    din = torch.empty((B * Hi * Wi, C), dtype=F32, device=dout.device)
    # separable two-pass form for the 4x / 8x resizes of wide tensors (the aux decoder's 512-channel maps)
    ws = torch.empty(B * Ho * Wi * C, dtype=F32, device=dout.device) if (C >= 64 and Ho == Wo and Hi == Wi and Ho // Hi in (4, 8) and Ho % Hi == 0) else None
    check(L.lib().mdv_upsample_bwd(ptr(dout), int(dout.dtype == BF16), ld_out or C, ptr(din), C, B, Hi, Wi, Ho, Wo, C, ptr(ws), L.stream()),
          "mdv_upsample_bwd")
    return din


def upsample_add(out, ins, B, Ho, Wo, C, ld_out=None):
    """out [B*Ho*Wo, C] fp32 += sum of the bilinear resizes of the fp32 maps `ins` = [(x [B*Hi*Wi, C], Hi, Wi)] (at most 3)."""
    args = []
    for x, Hi, Wi in list(ins) + [(None, 0, 0)] * (3 - len(ins)):
        args += [ptr(x), Hi, Wi]
    check(L.lib().mdv_upsample_add(ptr(out), ld_out or C, B, Ho, Wo, C, *args, L.stream()), "mdv_upsample_add")
    return out


class _MatmulDesc(ctypes.Structure):
    _fields_ = [("A", ctypes.c_void_p), ("B", ctypes.c_void_p), ("C", ctypes.c_void_p), ("u", ctypes.c_void_p), ("v", ctypes.c_void_p)] + \
               [(n, ctypes.c_int) for n in ("lda", "ldb", "ldc", "M", "N", "K", "trans_a", "trans_b", "accumulate", "pad_")]


def mm(A, B, C, M, N, K, *, lda=None, ldb=None, ldc=None, trans_a=False, trans_b=False, accumulate=False, u=None, v=None):
    """One problem of matmul_f32: C[M,N] (+)= op(A)[M,K] . op(B)[K,N] (+ u v^T), op = transpose when trans_*.  None when C is None
    (the gradient it would produce is off in this backward mode).  The descriptor holds references to its tensors until the
    launch: it carries raw device pointers, and a tensor freed before then could have its memory handed to the next one."""
    if C is None:
        return None
    d = _MatmulDesc(ptr(A), ptr(B), ptr(C), ptr(u), ptr(v), lda or (M if trans_a else K), ldb or (K if trans_b else N), ldc or N, M, N, K,
                    int(trans_a), int(trans_b), int(accumulate), 0)
    d.tensors = (A, B, C, u, v)
    return d


def matmul_f32(problems):
    """Independent fp32 products (mm(...) descriptors with distinct outputs; None entries skipped) in one launch."""
    ds = [d for d in problems if d is not None]
    if ds:
        check(L.lib().mdv_matmul_f32_grouped((_MatmulDesc * len(ds))(*ds), len(ds), L.stream()), "mdv_matmul_f32_grouped")


def _contig(t):
    return t if t.is_contiguous() else t.contiguous()


# Backward mode.  "all": every gradient (the default; what autograd expects).  "da_only": only the activation-gradient
# chain and the domain-adapter (`domain_layer`) gradients are computed — all other weight-gradient kernels are skipped.
# MKDTrainer's single-sweep schedule uses it for the aux-loss pass (train_step.py); see DESIGN.md "MKD backward schedule".
_BWD_MODE = "all"


class backward_mode:
    def __init__(self, mode):
        assert mode in ("all", "da_only")
        self.mode = mode

    def __enter__(self):
        global _BWD_MODE
        self.prev, _BWD_MODE = _BWD_MODE, self.mode

    def __exit__(self, *exc):
        global _BWD_MODE
        _BWD_MODE = self.prev


def wgrad_on():
    return _BWD_MODE == "all"


# Data-parallel bookkeeping hooks (train_step.GradBucketer).  Every Function remembers the tag that was current during
# its forward (the trainer tags each domain's forward) and reports the parameters it has just finished accumulating
# gradients for at the end of its backward, so the trainer can all-reduce a gradient bucket as soon as it is final.
_FWD_TAG = None
_FWD_USE_CB = None
_GRAD_READY_CB = None


def set_forward_tag(tag):
    global _FWD_TAG
    _FWD_TAG = tag


def set_forward_use_cb(cb):
    global _FWD_USE_CB
    _FWD_USE_CB = cb


def set_grad_ready_cb(cb):
    global _GRAD_READY_CB
    _GRAD_READY_CB = cb


def _fwd_mark(ctx):
    ctx.tag = _FWD_TAG
    if _FWD_USE_CB is not None:
        _FWD_USE_CB(_FWD_TAG, ctx.params)


def _grads_done(ctx):
    if _GRAD_READY_CB is not None:
        _GRAD_READY_CB(ctx.tag, ctx.params)


def enable_inplace_grad_accumulation(params, on=True):
    """Opt-in for gtarget()'s fast path: weight-gradient kernels of these parameters add straight into `p.grad` and
    backward returns None for them, i.e. autograd's AccumulateGrad node (tensor hooks, post-accumulate-grad hooks, a
    stock DDP/FSDP reducer, optimizer-in-backward) is BYPASSED.  Only a caller that owns the gradient buffers and the
    reduction may switch it on — train_step.MKDTrainer does, for its flat buffer.  Off by default: a plain
    `loss.backward()` / `torch.autograd.grad()` on the module behaves like any nn.Module."""
    for p in params:
        p._mdv_inplace_grad = bool(on)


def gtarget(p, shape=None, da=False):
    """Where a parameter gradient is accumulated.  Returns (buffer, value_to_return_from_backward).

    All parameter-gradient kernels ACCUMULATE (+=) into a zero-initialised buffer that backward returns, so autograd
    installs / accumulates it through AccumulateGrad like any other gradient (hooks fire, torch.autograd.grad works).
    Parameters opted in with enable_inplace_grad_accumulation() that already own a contiguous fp32 .grad get the kernels'
    sums added straight into it instead, and backward returns None for them.  A parameter whose requires_grad was switched
    off after the forward (multi_train_MDViT.py:198-200 freezes `domain_layer`) gets a scratch buffer and nothing is
    returned."""
    if p is None or (_BWD_MODE == "da_only" and not da):
        return None, None
    if not p.requires_grad:      # frozen after the forward: compute into scratch, hand nothing to autograd
        z = torch.zeros_like(p, memory_format=torch.contiguous_format)
        return (z if shape is None else z.view(shape)), None
    if getattr(p, "_mdv_inplace_grad", False):
        g = p.grad
        if g is not None and g.dtype == F32 and g.is_contiguous() and g.device == p.device and g.data_ptr() % 16 == 0:
            return (g if shape is None else g.view(shape)), None
    z = torch.zeros_like(p, memory_format=torch.contiguous_format)
    return (z if shape is None else z.view(shape)), z


def _dev_ctx(t):
    return torch.cuda.device(t.device)


# Fused fc1 -> GELU -> fc2 kernel for the widths it supports (C in {64,128}); MDV_NO_FUSED_MLP=1 keeps the two-GEMM path (A/B).
import os as _os
_FUSED_MLP = not bool(int(_os.environ.get("MDV_NO_FUSED_MLP", "0")))


# ------------------------------------------------------------------------------------------------- SerialBlock
class BlockFn(torch.autograd.Function):
    """SerialBlock_adapt.forward (mdvit.py:346-361) incl. ConvPosEnc, FactorAtt_ConvRelPosEnc(_Sup) and Mlp.  The trailing `norm`
    arguments are norm1 and norm2 of S sets (see _norm_slots)."""

    @staticmethod
    def forward(ctx, x, label, cpe_w, cpe_b, c3w, c3b, c5w, c5b, c7w, c7b, qkv_w, qkv_b, proj_w, proj_b,
                da_w1, da_b1, da_w2, da_b2, fc1_w, fc1_b, fc2_w, fc2_b, H, W, drop, dpr, training, *norm):
        B, N, C = x.shape
        M, dev = B * N, x.device
        hidden = fc1_w.shape[0]
        x = _contig(x)
        lib = L.lib()
        ctx.params = (cpe_w, cpe_b, c3w, c3b, c5w, c5b, c7w, c7b, qkv_w, qkv_b, proj_w, proj_b, da_w1, da_b1, da_w2, da_b2,
                      fc1_w, fc1_b, fc2_w, fc2_b) + norm
        (n1w, n1b), (n2w, n2b) = _norm_slots(norm, 2)
        _check_norm_sets(training)
        with _dev_ctx(x):
            x1 = dwconv3(x, cpe_w, cpe_b, B, H, W, H, W, C, 1, residual=True)
            ln1, mean1, rstd1 = layernorm_fwd(x1, n1w, n1b, M, C, rows_per_sample=N)
            qkv = torch.empty((M, 3 * C), dtype=BF16, device=dev)
            gemm_nt(ln1, prep_weight(qkv_w, 0, 3 * C, C), M, 3 * C, C, qkv, bias=qkv_b)
            gate = hid = None
            if label is not None and da_w1 is not None:
                label = _contig(label.float())
                nd, hd = da_w1.shape[1], da_w1.shape[0]
                gate = torch.empty((B, C), dtype=F32, device=dev)
                hid = torch.empty((B, hd), dtype=F32, device=dev)
                check(lib.mdv_da_gate_fwd(ptr(label), ptr(da_w1), ptr(da_b1), ptr(da_w2), ptr(da_b2), ptr(hid), ptr(gate), B, nd, hd,
                                          C, HEADS, L.stream()), "mdv_da_gate_fwd")
            stats = torch.empty(lib.mdv_attn_stats_floats(B, C, HEADS), dtype=F32, device=dev)
            ws = torch.empty(lib.mdv_attn_ws_floats(B, C, HEADS), dtype=F32, device=dev)
            y = torch.empty((M, C), dtype=BF16, device=dev)
            # dwconv(V)+b is kept for the backward pass (grad mode is always off inside Function.forward: ask ctx instead)
            ecrpe = torch.empty((M, C), dtype=BF16, device=dev) if any(ctx.needs_input_grad) else None
            check(lib.mdv_attn_fwd(ptr(qkv), ptr(gate), ptr(c3w), ptr(c3b), ptr(c5w), ptr(c5b), ptr(c7w), ptr(c7b), ptr(stats), ptr(ws),
                                   ptr(y), ptr(ecrpe), B, H, W, C, HEADS, L.stream()), "mdv_attn_fwd")
            p_drop = drop if training else 0.0
            sid = [new_stream_id() for _ in range(5)] if training and (drop > 0 or dpr > 0) else [0] * 5
            dp1 = dp2 = None
            if training and dpr > 0:
                dp1 = torch.empty(B, dtype=F32, device=dev)
                dp2 = torch.empty(B, dtype=F32, device=dev)
                rng = rng_tensor(dev)
                check(lib.mdv_droppath_scale(ptr(dp1), B, ctypes.c_float(dpr), ptr(rng), sid[3], L.stream()), "mdv_droppath_scale")
                check(lib.mdv_droppath_scale(ptr(dp2), B, ctypes.c_float(dpr), ptr(rng), sid[4], L.stream()), "mdv_droppath_scale")
            x2 = torch.empty((M, C), dtype=F32, device=dev)
            gemm_nt(y, prep_weight(proj_w, 0, C, C), M, C, C, x2, bias=proj_b, residual=x1, drop_p=p_drop, drop_stream=sid[0],
                    rowscale=dp1, rows_per_scale=N)
            ln2, mean2, rstd2 = layernorm_fwd(x2, n2w, n2b, M, C, rows_per_sample=N)
            need_grad = any(ctx.needs_input_grad)
            x3 = torch.empty((B, N, C), dtype=F32, device=dev)
            fused_mlp = bool(lib.mdv_mlp_supported(C, hidden)) and _FUSED_MLP
            if fused_mlp:
                # fc1 -> GELU -> dropout -> fc2 -> dropout -> DropPath -> + residual in ONE kernel: the hidden activation stays
                # on the SM (it is written out, with u, only when a backward pass will need them)
                u = torch.empty((M, hidden), dtype=BF16, device=dev) if need_grad else None
                hact = torch.empty((M, hidden), dtype=BF16, device=dev) if need_grad else None
                check(lib.mdv_mlp_fwd(ptr(ln2), ptr(prep_weight(fc1_w, 0, hidden, C)), ptr(fc1_b), ptr(prep_weight(fc2_w, 0, C, hidden)),
                                      ptr(fc2_b), ptr(x2), ptr(x3), ptr(hact), ptr(u), M, C, hidden, ctypes.c_float(p_drop),
                                      ptr(rng_tensor(dev)) if p_drop > 0 else None, sid[1], sid[2], ptr(dp2), N, L.stream()), "mdv_mlp_fwd")
            else:
                u = torch.empty((M, hidden), dtype=BF16, device=dev)
                hact = torch.empty((M, hidden), dtype=BF16, device=dev)
                # u receives gelu'(fc1 output) * dropout mask/(1-p): the factor the backward multiplies d(hact) by
                gemm_nt(ln2, prep_weight(fc1_w, 0, hidden, C), M, hidden, C, hact, bias=fc1_b, act=ACT_GELU, out_preact=u, drop_p=p_drop,
                        drop_stream=sid[1], preact_mode=1)
                gemm_nt(hact, prep_weight(fc2_w, 0, C, hidden), M, C, hidden, x3, bias=fc2_b, residual=x2, drop_p=p_drop,
                        drop_stream=sid[2], rowscale=dp2, rows_per_scale=N)
        ctx.save_for_backward(x, label, x1, mean1, rstd1, ln1, qkv, gate, hid, stats, y, x2, mean2, rstd2, ln2, u, hact, dp1, dp2, ecrpe)
        ctx.meta = (B, N, C, H, W, hidden, p_drop, sid, fused_mlp)
        _fwd_mark(ctx)
        return x3

    @staticmethod
    def backward(ctx, dx3):
        (x, label, x1, mean1, rstd1, ln1, qkv, gate, hid, stats, y, x2, mean2, rstd2, ln2, u, hact, dp1, dp2, ecrpe) = ctx.saved_tensors
        names = ("cpe_w", "cpe_b", "c3w", "c3b", "c5w", "c5b", "c7w", "c7b", "qkv_w", "qkv_b", "proj_w", "proj_b", "da_w1", "da_b1",
                 "da_w2", "da_b2", "fc1_w", "fc1_b", "fc2_w", "fc2_b")
        (cpe_w, cpe_b, c3w, c3b, c5w, c5b, c7w, c7b, qkv_w, qkv_b, proj_w, proj_b, da_w1, da_b1, da_w2, da_b2,
         fc1_w, fc1_b, fc2_w, fc2_b) = ctx.params[:20]
        norm = ctx.params[20:]
        B, N, C, H, W, hidden, p_drop, sid, fused_mlp = ctx.meta
        M, dev = B * N, x.device
        lib = L.lib()
        dx3 = _contig(dx3.float())
        T = {n: gtarget(p, da=n.startswith("da_")) for n, p in zip(names, ctx.params)}
        G = {k: v[0] for k, v in T.items()}
        TN = [gtarget(p) for p in norm]
        (n1w, _), (n2w, _) = _norm_slots(norm, 2)
        (G["n1w"], G["n1b"]), (G["n2w"], G["n2b"]) = _norm_slots([t[0] for t in TN], 2)
        with _dev_ctx(x):
            # ---- MLP
            # bias gradients (column sums) are by-products of the kernels that produce each output gradient
            d_fc2 = cast_bf16(dx3, M, C, rowscale=dp2, rows_per_scale=N, drop_p=p_drop, drop_stream=sid[2], colsum=G["fc2_b"])
            gemm_tn(d_fc2, hact, M, C, hidden, G["fc2_w"])
            dln2 = torch.empty((M, C), dtype=F32, device=dev)
            if fused_mlp:
                # du = (d_fc2 W2) * u and dln2 = du W1 in one kernel; du reaches HBM only when the fc1 weight gradient needs it
                du = torch.empty((M, hidden), dtype=BF16, device=dev) if G["fc1_w"] is not None else None
                check(lib.mdv_mlp_bwd(ptr(d_fc2), ptr(prep_weight(fc2_w, 1, C, hidden)), ptr(u), ptr(prep_weight(fc1_w, 1, hidden, C)),
                                      ptr(du), ptr(dln2), ptr(G["fc1_b"]), M, C, hidden, L.stream()), "mdv_mlp_bwd")
                if du is not None:
                    gemm_tn(du, ln2, M, hidden, C, G["fc1_w"])
            else:
                du = torch.empty((M, hidden), dtype=BF16, device=dev)
                gemm_nt(d_fc2, prep_weight(fc2_w, 1, C, hidden), M, hidden, C, du, mul_gelu_grad=u, mul_mode=1, colsum=G["fc1_b"])
                gemm_tn(du, ln2, M, hidden, C, G["fc1_w"])
                gemm_nt(du, prep_weight(fc1_w, 1, hidden, C), M, C, hidden, dln2)
            dx2, d_proj = layernorm_bwd(dln2, x2, mean2, rstd2, n2w, dx3, M, C, G["n2w"], G["n2b"], masked=True, rowscale=dp1,
                                        rows_per_scale=N, drop_p=p_drop, drop_stream=sid[0], dbias_masked=G["proj_b"])
            # ---- attention
            gemm_tn(d_proj, y, M, C, C, G["proj_w"])
            dy = torch.empty((M, C), dtype=BF16, device=dev)
            gemm_nt(d_proj, prep_weight(proj_w, 1, C, C), M, C, C, dy)
            dqkv = torch.empty((M, 3 * C), dtype=BF16, device=dev)
            Ch = C // HEADS
            da_live = gate is not None and da_w1.requires_grad and da_w2.requires_grad
            dgate = torch.empty((B, C), dtype=F32, device=dev) if gate is not None else None      # (zeroed by mdv_attn_bwd)
            ws = torch.empty(lib.mdv_attn_ws_floats(B, C, HEADS), dtype=F32, device=dev)
            check(lib.mdv_attn_bwd(ptr(qkv), ptr(dy), ptr(y), ptr(ecrpe), ptr(gate), ptr(c3w), ptr(c3b), ptr(c5w), ptr(c5b), ptr(c7w), ptr(c7b),
                                   ptr(stats), ptr(dqkv), ptr(dgate), ptr(G["c3w"]), ptr(G["c3b"]), ptr(G["c5w"]), ptr(G["c5b"]),
                                   ptr(G["c7w"]), ptr(G["c7b"]), ptr(G["qkv_b"]), ptr(ws), B, H, W, C, HEADS, L.stream()), "mdv_attn_bwd")
            if da_live:
                nd, hd = da_w1.shape[1], da_w1.shape[0]
                ws2 = torch.empty(B * (C + hd), dtype=F32, device=dev)
                check(lib.mdv_da_gate_bwd(ptr(label), ptr(da_w2), ptr(hid), ptr(gate), ptr(dgate), ptr(G["da_w1"]), ptr(G["da_b1"]),
                                          ptr(G["da_w2"]), ptr(G["da_b2"]), ptr(ws2), B, nd, hd, C, HEADS, L.stream()), "mdv_da_gate_bwd")
            gemm_tn(dqkv, ln1, M, 3 * C, C, G["qkv_w"])        # (qkv bias gradient: by-product of mdv_attn_bwd)
            dln1 = torch.empty((M, C), dtype=F32, device=dev)
            gemm_nt(dqkv, prep_weight(qkv_w, 1, 3 * C, C), M, C, 3 * C, dln1)
            dx1, _ = layernorm_bwd(dln1, x1, mean1, rstd1, n1w, dx2, M, C, G["n1w"], G["n1b"])
            # ---- ConvPosEnc
            dx = dwconv3(dx1, cpe_w, None, B, H, W, H, W, C, 1, transposed=True, residual=True)
            dwconv3_wgrad(dx1, x, G["cpe_w"], G["cpe_b"], B, H, W, H, W, C, 1)
        _grads_done(ctx)
        return (dx.view(B, N, C), None, *(T[n][1] for n in names), None, None, None, None, None, *(t[1] for t in TN))


# ------------------------------------------------------------------------------------------------- conv pieces
def _bn_args(bn):
    return bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.num_batches_tracked


# The norm Functions below (and BlockFn) take the norm parameters of S sets as trailing tensor arguments `norm` (autograd only
# tracks direct tensor arguments): set by set, and within a set the Function's k norm slots in order, each as (weight, bias).
# Their `bufs` hold each set's running buffers in the same order, (running_mean, running_var, num_batches_tracked) per slot.
# S = 1 is a plain module; S > 1 is the stacked pass of the domain-specific-norm models, where row group g uses set g
# (model._norm_args builds both).
def _norm_slots(norm, k, bufs=()):
    """Per-slot lists over the S sets: k lists [weights, biases], extended by [running_means, running_vars, nbts] when bufs are
    given."""
    slots = [[list(norm[2 * j + i::2 * k]) for i in range(2)] for j in range(k)]
    if bufs:
        for j, sl in enumerate(slots):
            sl += [list(bufs[3 * j + i::3 * k]) for i in range(3)]
    return slots


def _norm_grads(*slots):
    """The values backward returns for the trailing norm arguments: slots = each slot's (weight grads, bias grads) lists over the
    sets, flattened in _norm_slots' order."""
    return tuple(r for s in range(len(slots[0][0])) for gw, gb in slots for r in (gw[s], gb[s]))


def _conv_bn_fwd(A, w, M, K, slot, act, training, rows_per_sample, conv_bias=None):
    """One conv -> BatchNorm -> act stage of the MDViT conv trunk: a TF32 GEMM of the fp32 operand A [M, K] (the im2col matrix of a
    3x3 conv in mdv_im2col3 order, padded to K columns, or the input of a 1x1 conv) with the conv weight w [Cout, Cin, k, k].
    slot = (weights, biases, running_means, running_vars, nbts), lists over the S norm sets (_norm_slots).
    Training: the GEMM writes z = conv + conv_bias, and bn_forward normalises each bn_groups() row group with its batch statistics.
    Eval: the running statistics and conv_bias fold into the GEMM epilogue (bn_fold), so z never reaches HBM; inside norm_sets with
    S > 1, row m takes the folded set of sample sample_set[m // rows_per_sample].
    Returns (y [M, Cout] fp32, (z, mean, rstd) to save for backward; all None in eval)."""
    g, b, rm, rv, nb = slot
    _check_norm_sets(training)
    if not training:
        scale, shift = bn_fold(g, b, rm, rv, conv_bias)
    Cout, Cin = w.shape[:2]
    Wt = prep_weight(w, 2 | 8, Cout, 9 * Cin, ld=K, cin=Cin) if w.shape[2] == 3 else _contig(w).view(Cout, K)
    out = torch.empty((M, Cout), dtype=F32, device=A.device)
    if training:
        gemm_nt(A, Wt, M, Cout, K, out, bias=conv_bias, tf32=True)
        y, mean, rstd = bn_forward(out, M, Cout, g, b, rm, rv, nb, training, act, False)
        return y, (out, mean, rstd)
    gemm_nt(A, Wt, M, Cout, K, out, tf32=True, colscale=scale, bias=shift, act=act, sample_set=_NORM_SETS if scale.dim() == 2 else None,
            rows_per_sample=rows_per_sample)
    return out, (None, None, None)


def _conv1_wgrad(dz, a, w):
    """Weight gradient of a 1x1 conv w [Cout, Cin, 1, 1] from dz [M, Cout] and its input a [M, Cin]; an fp32 a is cast to the bf16
    operand only when the gradient is wanted.  Returns what backward returns for w."""
    Cout, Cin = w.shape[:2]
    gw, rw = gtarget(w, (Cout, Cin))
    if gw is not None:
        M = dz.shape[0]
        gemm_tn(dz, a if a.dtype == BF16 else cast_bf16(a, M, Cin), M, Cout, Cin, gw)
    return rw


def _conv3_wgrad(dz, col, w):
    """Weight gradient of a 3x3 conv w [Cout, Cin, 3, 3] from dz [M, Cout] and its im2col matrix col [M, ld] ((tap, channel) column
    order, ld >= 9 Cin; fp32 is cast to the bf16 operand only when the gradient is wanted): gemm_tn into a zeroed [Cout, ld] buffer,
    unpermuted into w's layout.  Returns what backward returns for w."""
    gw, rw = gtarget(w)
    if gw is not None:
        (M, ld), Cout, Cin = col.shape, w.shape[0], w.shape[1]
        gwp = gemm_tn(dz, col if col.dtype == BF16 else cast_bf16(col, M, ld), M, Cout, ld, torch.zeros((Cout, ld), dtype=F32, device=dz.device))
        check(L.lib().mdv_unperm_conv_grad(ptr(gwp), ld, ptr(gw), Cout, Cin, L.stream()), "mdv_unperm_conv_grad")
    return rw


def _conv3_bwd(dz, col, w, cb, B, H, W, Ho, Wo, stride):
    """Backward of a 3x3 conv (padding 1, stride `stride`, [B, H, W, Cin] -> [B, Ho, Wo, Cout]) run as im2col matrix col
    [B*Ho*Wo, 9 Cin] times w^T, plus conv bias cb (or None).  Returns (w's gradient, cb's gradient, dx [B*H*W, Cin] fp32)."""
    Cout, Cin = w.shape[:2]
    M, dev = dz.shape[0], dz.device
    rw = _conv3_wgrad(dz, col, w)
    gb, rb = gtarget(cb)
    colsum(dz, M, Cout, gb)
    dcol = gemm_nt(dz, prep_weight(w, 3, Cout, 9 * Cin, cin=Cin), M, 9 * Cin, Cout, torch.empty((M, 9 * Cin), dtype=F32, device=dev))
    dx = torch.empty((B * H * W, Cin), dtype=F32, device=dev)
    check(L.lib().mdv_col2im3(ptr(dcol), ptr(dx), B, H, W, Ho, Wo, Cin, stride, 9 * Cin, L.stream()), "mdv_col2im3")
    return rw, rb, dx


class StemFn(torch.autograd.Function):
    """stem = 2x (Conv3x3 s2 no-bias -> BN -> Hardswish), mdvit.py:509-526.  im2col (bf16) + tcgen05 GEMM."""

    @staticmethod
    def forward(ctx, img, w0, w1, bufs, training, *norm):
        B, _, H, W = img.shape
        dev = img.device
        img = _contig(img.float())
        H1, W1, H2, W2 = H // 2, W // 2, H // 4, W // 4
        M0, M1 = B * H1 * W1, B * H2 * W2
        ctx.params = (w0, w1) + norm
        slot0, slot1 = _norm_slots(norm, 2, bufs)
        lib = L.lib()
        with _dev_ctx(img):
            # TF32 operands (fp32 in memory) for both stem convs: see mdv_gemm_nt_tf32
            col0 = torch.empty((M0, 32), dtype=F32, device=dev)
            check(lib.mdv_im2col_stem(ptr(img), ptr(col0), 0, B, H, W, L.stream()), "mdv_im2col_stem")
            a0, saved0 = _conv_bn_fwd(col0, w0, M0, 32, slot0, ACT_HSWISH, training, H1 * W1)
            col1 = torch.empty((M1, 288), dtype=F32, device=dev)
            check(lib.mdv_im2col3(ptr(a0), 0, ptr(col1), 0, B, H1, W1, H2, W2, 32, 2, 288, L.stream()), "mdv_im2col3")
            y, saved1 = _conv_bn_fwd(col1, w1, M1, 288, slot1, ACT_HSWISH, training, H2 * W2)
        ctx.save_for_backward(col0, *saved0, col1, *saved1)
        ctx.meta = (B, H1, W1, H2, W2, training)
        _fwd_mark(ctx)
        ctx.set_materialize_grads(False)
        return y.view(B, H2 * W2, 64)

    @staticmethod
    def backward(ctx, dy):
        if dy is None:       # the da_only pass stops at the first patch embedding
            return (None,) * (3 + len(ctx.params))
        B, H1, W1, H2, W2, training = ctx.meta
        _require_train_bn(training)
        col0, z0, mean0, rstd0, col1, z1, mean1, rstd1 = ctx.saved_tensors
        w0, w1 = ctx.params[:2]
        (g0, b0), (g1, b1) = _norm_slots(ctx.params[2:], 2)
        dy = _contig(dy.float())
        with _dev_ctx(dy):
            dz1, rg1, rb1 = bn_backward(dy, z1, mean1, rstd1, g1, b1, ACT_HSWISH, B * H2 * W2, 64)
            rw1, _, da0 = _conv3_bwd(dz1, col1, w1, None, B, H1, W1, H2, W2, 2)
            dz0, rg0, rb0 = bn_backward(da0, z0, mean0, rstd0, g0, b0, ACT_HSWISH, B * H1 * W1, 32)
            rw0 = _conv3_wgrad(dz0, col0, w0)
        _grads_done(ctx)
        return (None, rw0, rw1, None, None) + _norm_grads((rg0, rb0), (rg1, rb1))


class PatchEmbedFn(torch.autograd.Function):
    """DWCPatchEmbed: depthwise 3x3 (stride s) -> 1x1 conv -> BN -> Hardswish, mdvit.py:114-123."""

    @staticmethod
    def forward(ctx, x, dw_w, pw_w, bufs, Hi, Wi, stride, training, after_stem, *norm):
        B, _, Cin = x.shape
        C = pw_w.shape[0]
        Ho, Wo = (Hi + 2 - 3) // stride + 1, (Wi + 2 - 3) // stride + 1
        M = B * Ho * Wo
        x = _contig(x)
        ctx.params = (dw_w, pw_w) + norm
        (slot,) = _norm_slots(norm, 1, bufs)
        with _dev_ctx(x):
            t = dwconv3(x, dw_w, None, B, Hi, Wi, Ho, Wo, Cin, stride)          # fp32: TF32 operand of the pointwise conv
            y, (z, mean, rstd) = _conv_bn_fwd(t, pw_w, M, Cin, slot, ACT_HSWISH, training, Ho * Wo)
        ctx.save_for_backward(x, t, z, mean, rstd)
        ctx.meta = (B, Hi, Wi, Ho, Wo, Cin, C, stride, training)
        _fwd_mark(ctx)
        ctx.after_stem = after_stem
        return y.view(B, Ho * Wo, C)

    @staticmethod
    def backward(ctx, dy):
        B, Hi, Wi, Ho, Wo, Cin, C, stride, training = ctx.meta
        _require_train_bn(training)
        x, t, z, mean, rstd = ctx.saved_tensors
        dw_w, pw_w = ctx.params[:2]
        ((g, b),) = _norm_slots(ctx.params[2:], 1)
        if ctx.after_stem and not wgrad_on():
            # nothing upstream of the first patch embedding owns a domain adapter: the da_only pass stops here
            return (None,) * (7 + len(ctx.params))
        M, dev = B * Ho * Wo, dy.device
        dy = _contig(dy.float())
        with _dev_ctx(dy):
            dz, rg, rb = bn_backward(dy, z, mean, rstd, g, b, ACT_HSWISH, M, C)
            r_pw = _conv1_wgrad(dz, t, pw_w)
            dt = torch.empty((M, Cin), dtype=F32, device=dev)
            gemm_nt(dz, prep_weight(pw_w, 1, C, Cin), M, Cin, C, dt)
            dx = dwconv3(dt, dw_w, None, B, Ho, Wo, Hi, Wi, Cin, stride, transposed=True)
            g_dw, r_dw = gtarget(dw_w)
            dwconv3_wgrad(dt, x, g_dw, None, B, Hi, Wi, Ho, Wo, Cin, stride)
        _grads_done(ctx)
        return (dx.view(B, Hi * Wi, Cin), r_dw, r_pw, None, None, None, None, None, None) + _norm_grads((rg, rb))


class BridgeFn(torch.autograd.Function):
    """bridge = 2x (Conv3x3 + bias -> BN -> ReLU), mdvit.py:557-564."""

    @staticmethod
    def forward(ctx, x, w0, c0, w1, c1, bufs, H, W, training, *norm):
        B, _, C = x.shape
        C0, C1 = w0.shape[0], w1.shape[0]
        M, dev = B * H * W, x.device
        x = _contig(x)
        ctx.params = (w0, c0, w1, c1) + norm
        slot0, slot1 = _norm_slots(norm, 2, bufs)
        lib = L.lib()
        with _dev_ctx(x):
            col0 = torch.empty((M, 9 * C), dtype=F32, device=dev)
            check(lib.mdv_im2col3(ptr(x), 0, ptr(col0), 0, B, H, W, H, W, C, 1, 9 * C, L.stream()), "mdv_im2col3")
            col1 = torch.empty((M, 9 * C0), dtype=F32, device=dev)
            a0, saved0 = _conv_bn_fwd(col0, w0, M, 9 * C, slot0, ACT_RELU, training, H * W, c0)
            check(lib.mdv_im2col3(ptr(a0), 0, ptr(col1), 0, B, H, W, H, W, C0, 1, 9 * C0, L.stream()), "mdv_im2col3")
            y, saved1 = _conv_bn_fwd(col1, w1, M, 9 * C0, slot1, ACT_RELU, training, H * W, c1)
        ctx.save_for_backward(col0, *saved0, col1, *saved1)
        ctx.meta = (B, H, W, C, C0, C1, training)
        _fwd_mark(ctx)
        return y.view(B, H * W, C1)

    @staticmethod
    def backward(ctx, dy):
        B, H, W, C, C0, C1, training = ctx.meta
        _require_train_bn(training)
        col0, z0, mean0, rstd0, col1, z1, mean1, rstd1 = ctx.saved_tensors
        w0, c0, w1, c1 = ctx.params[:4]
        (g0, b0), (g1, b1) = _norm_slots(ctx.params[4:], 2)
        M = B * H * W
        dy = _contig(dy.float())
        with _dev_ctx(dy):
            dz1, rg1, rb1 = bn_backward(dy, z1, mean1, rstd1, g1, b1, ACT_RELU, M, C1)
            rw1, rc1, da0 = _conv3_bwd(dz1, col1, w1, c1, B, H, W, H, W, 1)
            dz0, rg0, rb0 = bn_backward(da0, z0, mean0, rstd0, g0, b0, ACT_RELU, M, C0)
            rw0, rc0, dx = _conv3_bwd(dz0, col0, w0, c0, B, H, W, H, W, 1)
        _grads_done(ctx)
        return (dx.view(B, H * W, C), rw0, rc0, rw1, rc1, None, None, None, None) + _norm_grads((rg0, rb0), (rg1, rb1))


class DecoderConvFn(torch.autograd.Function):
    """Conv part of UnetDecodingBlockTransformer.forward (Decoders.py:194-205): bilinear up -> 1x1 conv_before -> cat(skip, .) ->
    grouped 3x3 (2 in/group) -> 1x1 -> BN -> Hardswish.  conv_before is commuted in front of the resize (exact)."""

    @staticmethod
    def forward(ctx, inp, skip, cb_w, cb_b, dw_w, pw_w, bufs, h, w, H, W, training, *norm):
        B, _, Cin = inp.shape
        C = cb_w.shape[0]
        m, M, dev = B * h * w, B * H * W, inp.device
        inp, skip = _contig(inp), _contig(skip)
        ctx.params = (cb_w, cb_b, dw_w, pw_w) + norm
        (slot,) = _norm_slots(norm, 1, bufs)
        lib = L.lib()
        with _dev_ctx(inp):
            # both 1x1 convs of the decoder trunk run on TF32 operands (fp32 in memory): see mdv_gemm_nt_tf32
            t = torch.empty((m, C), dtype=F32, device=dev)
            gemm_nt(inp.view(m, Cin), _contig(cb_w).view(C, Cin), m, C, Cin, t, bias=cb_b, tf32=True)
            up = upsample_fwd(t, torch.empty((M, C), dtype=F32, device=dev), B, h, w, H, W, C)
            gc = torch.empty((M, C), dtype=F32, device=dev)
            check(lib.mdv_gconv2_fwd(ptr(skip), ptr(up), ptr(dw_w), ptr(gc), 0, B, H, W, C, L.stream()), "mdv_gconv2_fwd")
            y, (z, mean, rstd) = _conv_bn_fwd(gc, pw_w, M, C, slot, ACT_HSWISH, training, H * W)
        ctx.save_for_backward(skip, inp, up, gc, z, mean, rstd)
        ctx.meta = (B, h, w, H, W, Cin, C, training)
        _fwd_mark(ctx)
        return y.view(B, H * W, C)

    @staticmethod
    def backward(ctx, dy):
        B, h, w, H, W, Cin, C, training = ctx.meta
        _require_train_bn(training)
        skip, inp, up, gc, z, mean, rstd = ctx.saved_tensors
        cb_w, cb_b, dw_w, pw_w = ctx.params[:4]
        ((g, b),) = _norm_slots(ctx.params[4:], 1)
        m, M, dev = B * h * w, B * H * W, dy.device
        lib = L.lib()
        dy = _contig(dy.float())
        with _dev_ctx(dy):
            dz, rg, rb = bn_backward(dy, z, mean, rstd, g, b, ACT_HSWISH, M, C)
            r_pw = _conv1_wgrad(dz, gc, pw_w)
            dgc = torch.empty((M, C), dtype=F32, device=dev)
            gemm_nt(dz, prep_weight(pw_w, 1, C, C), M, C, C, dgc)
            dskip = torch.empty((M, C), dtype=F32, device=dev)
            dup = torch.empty((M, C), dtype=F32, device=dev)
            g_dw, r_dw = gtarget(dw_w)
            check(lib.mdv_gconv2_bwd(ptr(dgc), ptr(skip), ptr(up), ptr(dw_w), ptr(dskip), ptr(dup), ptr(g_dw), B, H, W, C, L.stream()),
                  "mdv_gconv2_bwd")
            dt = upsample_bwd(dup, B, h, w, H, W, C)
            dtb = cast_bf16(dt, m, C)
            r_cb = _conv1_wgrad(dtb, inp, cb_w)
            g_cbb, r_cbb = gtarget(cb_b)
            colsum(dt, m, C, g_cbb)
            dinp = torch.empty((m, Cin), dtype=F32, device=dev)
            gemm_nt(dtb, prep_weight(cb_w, 1, C, Cin), m, Cin, C, dinp)
        _grads_done(ctx)
        return ((dinp.view(B, h * w, Cin), dskip.view(B, H * W, C), r_cb, r_cbb, r_dw, r_pw, None, None, None, None, None, None)
                + _norm_grads((rg, rb)))


def _sum_tokens(t, B, H, W, C):
    """[B, H*W, C] -> [B, C] sums over the tokens of each image: the exact transpose of the 1x1 -> HxW bilinear resize."""
    out = torch.empty((B, C), dtype=F32, device=t.device)
    check(L.lib().mdv_upsample_bwd(ptr(t), int(t.dtype == BF16), C, ptr(out), C, B, 1, 1, H, W, C, None, L.stream()), "mdv_upsample_bwd")
    return out


class DeepLabFn(torch.autograd.Function):
    """DeepLabV3Decoder.classifier[0:4] (Decoders.py:218-227, Utils/_deeplab.py:115-166) on token-major input: ASPP (1x1 conv,
    three dilated 3x3 convs, image pooling; each conv -> BN -> ReLU) -> concat -> 1x1 project -> BN -> ReLU -> Dropout(0.1) ->
    3x3 conv -> BN -> ReLU.  The final 1x1 conv + bilinear resize is ops.HeadFn.  Every conv is an (im2col +) tcgen05 GEMM with
    bf16 operands; the branch outputs are written straight into their column slice of the concat buffer.  The maps are tiny
    (H/32 x W/32), so this Function is written for coverage, not speed."""

    NB = 7      # conv+BN pairs: aspp 1x1, 3 dilated, pooling, project, 3x3

    @staticmethod
    def forward(ctx, x, H, W, dils, drop_p, training, bufs, *wgb):
        B, N, Cin = x.shape
        M, dev = B * N, x.device
        x = _contig(x)
        ws, gs, bs = wgb[0::3], wgb[1::3], wgb[2::3]
        Co = ws[0].shape[0]
        lib = L.lib()
        sid = new_stream_id() if (training and drop_p > 0) else 0
        saved = {}

        def bn(k, z, rows):
            rm, rv, nb = bufs[k]
            y, mean, rstd = bn_forward(z, rows, Co, [gs[k]], [bs[k]], [rm], [rv], [nb], training, ACT_RELU, False)
            saved[k] = (z, mean, rstd)
            return y

        with _dev_ctx(x):
            xb = cast_bf16(x, M, Cin)
            cat = torch.empty((M, 5 * Co), dtype=BF16, device=dev)
            # 1x1 branch
            z = gemm_nt(xb, prep_weight(ws[0], 0, Co, Cin), M, Co, Cin, torch.empty((M, Co), dtype=F32, device=dev))
            cast_bf16(bn(0, z, M), M, Co, out=cat[:, 0:Co], ld_out=5 * Co)
            # dilated 3x3 branches
            col = torch.empty((M, 9 * Cin), dtype=BF16, device=dev)
            for k in (1, 2, 3):
                check(lib.mdv_im2col3_dil(ptr(xb), 1, ptr(col), B, H, W, Cin, int(dils[k - 1]), 9 * Cin, L.stream()), "mdv_im2col3_dil")
                z = gemm_nt(col, prep_weight(ws[k], 2, Co, 9 * Cin, cin=Cin), M, Co, 9 * Cin, torch.empty((M, Co), dtype=F32, device=dev))
                cast_bf16(bn(k, z, M), M, Co, out=cat[:, k * Co:(k + 1) * Co], ld_out=5 * Co)
            # image pooling: mean over the tokens of an image (the transpose of a 1x1 -> HxW resize is the sum), 1x1 conv, BN over the
            # B pooled rows, ReLU, broadcast back (bilinear resize from 1x1)
            inv_n = torch.full((B,), 1.0 / N, dtype=F32, device=dev)
            pooled = cast_bf16(_sum_tokens(x, B, H, W, Cin), B, Cin, rowscale=inv_n, rows_per_scale=1)
            z = gemm_nt(pooled, prep_weight(ws[4], 0, Co, Cin), B, Co, Cin, torch.empty((B, Co), dtype=F32, device=dev))
            upsample_fwd(bn(4, z, B), cat[:, 4 * Co:], B, 1, 1, H, W, Co, ld_out=5 * Co)
            # project + dropout
            z = gemm_nt(cat, prep_weight(ws[5], 0, Co, 5 * Co), M, Co, 5 * Co, torch.empty((M, Co), dtype=F32, device=dev))
            pj = cast_bf16(bn(5, z, M), M, Co, drop_p=drop_p if training else 0.0, drop_stream=sid)
            # 3x3 conv
            col2 = torch.empty((M, 9 * Co), dtype=BF16, device=dev)
            check(lib.mdv_im2col3_dil(ptr(pj), 1, ptr(col2), B, H, W, Co, 1, 9 * Co, L.stream()), "mdv_im2col3_dil")
            z = gemm_nt(col2, prep_weight(ws[6], 2, Co, 9 * Co, cin=Co), M, Co, 9 * Co, torch.empty((M, Co), dtype=F32, device=dev))
            y = bn(6, z, M)
        ctx.meta = (B, N, Cin, Co, H, W, tuple(int(d) for d in dils), float(drop_p), sid, training)
        if training:
            flat = []
            for k in range(DeepLabFn.NB):
                flat += list(saved[k])
            ctx.save_for_backward(xb, pooled, cat, col2, *flat)
        ctx.params = tuple(wgb)
        _fwd_mark(ctx)
        return y.view(B, N, Co)

    @staticmethod
    def backward(ctx, dy):
        B, N, Cin, Co, H, W, dils, drop_p, sid, training = ctx.meta
        _require_train_bn(training)
        xb, pooled, cat, col2, *flat = ctx.saved_tensors
        wgb = ctx.params
        ws, gs, bs = wgb[0::3], wgb[1::3], wgb[2::3]
        M, dev = B * N, dy.device
        lib = L.lib()
        dy = _contig(dy.float())
        rets = [None] * (3 * DeepLabFn.NB)

        def bn_bwd(k, d, rows):
            z, mean, rstd = flat[3 * k:3 * k + 3]
            dz, (rg,), (rb,) = bn_backward(d, z, mean, rstd, [gs[k]], [bs[k]], ACT_RELU, rows, Co)
            rets[3 * k + 1], rets[3 * k + 2] = rg, rb
            return dz

        with _dev_ctx(dy):
            # 3x3 conv
            dz = bn_bwd(6, dy, M)
            rets[3 * 6] = _conv3_wgrad(dz, col2, ws[6])
            dcol = gemm_nt(dz, prep_weight(ws[6], 3, Co, 9 * Co, cin=Co), M, 9 * Co, Co, torch.empty((M, 9 * Co), dtype=F32, device=dev))
            dpj = torch.empty((M, Co), dtype=F32, device=dev)
            check(lib.mdv_col2im3_dil(ptr(dcol), ptr(dpj), B, H, W, Co, 1, 9 * Co, 0, L.stream()), "mdv_col2im3_dil")
            if drop_p > 0:      # the forward's mask, regenerated from the same counter stream
                dpj = cast_bf16(dpj, M, Co, drop_p=drop_p, drop_stream=sid).float()
            # project
            dz = bn_bwd(5, dpj, M)
            rets[3 * 5] = _conv1_wgrad(dz, cat, ws[5])
            wt = prep_weight(ws[5], 1, Co, 5 * Co)                       # [5 Co, Co]: rows = input channels of the concat

            def dcat(k):      # gradient of branch k's slice of the concat (contiguous)
                return gemm_nt(dz, wt[k * Co:(k + 1) * Co], M, Co, Co, torch.empty((M, Co), dtype=F32, device=dev))

            # image pooling: the broadcast's transpose sums over the tokens of an image
            dzp = bn_bwd(4, _sum_tokens(dcat(4), B, H, W, Co), B)
            rets[3 * 4] = _conv1_wgrad(dzp, pooled, ws[4])
            inv_n = torch.full((B,), 1.0 / N, dtype=F32, device=dev)
            dpool = gemm_nt(dzp, prep_weight(ws[4], 1, Co, Cin), B, Cin, Co, torch.empty((B, Cin), dtype=F32, device=dev), rowscale=inv_n,
                            rows_per_scale=1)
            dx = upsample_fwd(dpool, torch.empty((M, Cin), dtype=F32, device=dev), B, 1, 1, H, W, Cin)
            # dilated branches (the im2col matrices are rebuilt instead of saved)
            col = torch.empty((M, 9 * Cin), dtype=BF16, device=dev)
            dcolk = torch.empty((M, 9 * Cin), dtype=F32, device=dev)
            for k in (1, 2, 3):
                dzk = bn_bwd(k, dcat(k), M)
                if wgrad_on():
                    check(lib.mdv_im2col3_dil(ptr(xb), 1, ptr(col), B, H, W, Cin, dils[k - 1], 9 * Cin, L.stream()), "mdv_im2col3_dil")
                rets[3 * k] = _conv3_wgrad(dzk, col, ws[k])
                gemm_nt(dzk, prep_weight(ws[k], 3, Co, 9 * Cin, cin=Cin), M, 9 * Cin, Co, dcolk)
                check(lib.mdv_col2im3_dil(ptr(dcolk), ptr(dx), B, H, W, Cin, dils[k - 1], 9 * Cin, 1, L.stream()), "mdv_col2im3_dil")
            # 1x1 branch: dx += dz0 . W0
            dz0 = bn_bwd(0, dcat(0), M)
            rets[3 * 0] = _conv1_wgrad(dz0, xb, ws[0])
            gemm_nt(dz0, prep_weight(ws[0], 1, Co, Cin), M, Cin, Co, dx, residual=dx)
        _grads_done(ctx)
        return (dx.view(B, N, Cin), None, None, None, None, None, None, *rets)


class SdpaAttentionFn(torch.autograd.Function):
    """Attention_Sup.forward / Attention.forward of TransFuse_S_adapt's DeiT branch (vision_transformer.py:110-122,149-169):
    qkv Linear -> softmax(s Q K^T) V -> DA head gate -> proj Linear, as bf16 tcgen05 GEMMs around mdv_sdpa_fwd / mdv_sdpa_bwd.
    head_dim 64, N in {128, 256}; attn_drop = proj_drop = 0 (the reference's DeiT-S setting)."""

    @staticmethod
    def forward(ctx, x, label, qkv_w, qkv_b, proj_w, proj_b, da_w1, da_b1, da_w2, da_b2, heads, scale):
        B, N, C = x.shape
        M, dev = B * N, x.device
        x = _contig(x)
        lib = L.lib()
        with _dev_ctx(x):
            xb = cast_bf16(x, M, C)
            qkv = torch.empty((M, 3 * C), dtype=BF16, device=dev)
            gemm_nt(xb, prep_weight(qkv_w, 0, 3 * C, C), M, 3 * C, C, qkv, bias=qkv_b)
            gate = hid = None
            if da_w1 is not None:
                label = _contig(label.float())
                nd, hd = da_w1.shape[1], da_w1.shape[0]
                gate = torch.empty((B, C), dtype=F32, device=dev)
                hid = torch.empty((B, hd), dtype=F32, device=dev)
                check(lib.mdv_da_gate_fwd(ptr(label), ptr(da_w1), ptr(da_b1), ptr(da_w2), ptr(da_b2), ptr(hid), ptr(gate), B, nd, hd, C, heads,
                                          L.stream()), "mdv_da_gate_fwd")
            y = torch.empty((M, C), dtype=BF16, device=dev)
            lse = torch.empty((B, heads, N), dtype=F32, device=dev)
            check(lib.mdv_sdpa_fwd(ptr(qkv), ptr(gate), ptr(y), ptr(lse), B, N, C, heads, ctypes.c_float(scale), L.stream()), "mdv_sdpa_fwd")
            out = torch.empty((M, C), dtype=F32, device=dev)
            gemm_nt(y, prep_weight(proj_w, 0, C, C), M, C, C, out, bias=proj_b)
        ctx.save_for_backward(xb, qkv, y, lse, gate, hid, label if da_w1 is not None else None)
        ctx.params = (qkv_w, qkv_b, proj_w, proj_b, da_w1, da_b1, da_w2, da_b2)
        ctx.meta = (B, N, C, heads, float(scale))
        _fwd_mark(ctx)
        return out.view(B, N, C)

    @staticmethod
    def backward(ctx, dout):
        B, N, C, heads, scale = ctx.meta
        xb, qkv, y, lse, gate, hid, label = ctx.saved_tensors
        qkv_w, qkv_b, proj_w, proj_b, da_w1, da_b1, da_w2, da_b2 = ctx.params
        M, dev = B * N, dout.device
        lib = L.lib()
        dout = _contig(dout.float())
        with _dev_ctx(dout):
            dob = cast_bf16(dout, M, C)
            g_pw, r_pw = gtarget(proj_w)
            gemm_tn(dob, y, M, C, C, g_pw)
            g_pb, r_pb = gtarget(proj_b)
            colsum(dout, M, C, g_pb)
            dy = torch.empty((M, C), dtype=BF16, device=dev)
            gemm_nt(dob, prep_weight(proj_w, 1, C, C), M, C, C, dy)
            dqkv = torch.empty((M, 3 * C), dtype=BF16, device=dev)
            dgate = torch.empty((B, C), dtype=F32, device=dev) if gate is not None else None
            check(lib.mdv_sdpa_bwd(ptr(qkv), ptr(gate), ptr(y), ptr(lse), ptr(dy), ptr(dqkv), ptr(dgate), B, N, C, heads, ctypes.c_float(scale),
                                   L.stream()), "mdv_sdpa_bwd")
            r_da = [None] * 4
            if gate is not None:
                tg = [gtarget(p, da=True) for p in (da_w1, da_b1, da_w2, da_b2)]
                if tg[0][0] is not None:
                    nd, hd = da_w1.shape[1], da_w1.shape[0]
                    ws2 = torch.empty(B * (C + hd), dtype=F32, device=dev)
                    check(lib.mdv_da_gate_bwd(ptr(label), ptr(da_w2), ptr(hid), ptr(gate), ptr(dgate), ptr(tg[0][0]), ptr(tg[1][0]), ptr(tg[2][0]),
                                              ptr(tg[3][0]), ptr(ws2), B, nd, hd, C, heads, L.stream()), "mdv_da_gate_bwd")
                r_da = [t[1] for t in tg]
            g_qw, r_qw = gtarget(qkv_w)
            gemm_tn(dqkv, xb, M, 3 * C, C, g_qw)
            g_qb, r_qb = gtarget(qkv_b)
            colsum(dqkv, M, 3 * C, g_qb)
            dx = torch.empty((M, C), dtype=F32, device=dev)
            gemm_nt(dqkv, prep_weight(qkv_w, 1, 3 * C, C), M, C, 3 * C, dx)
        _grads_done(ctx)
        return (dx.view(B, N, C), None, r_qw, r_qb, r_pw, r_pb, *r_da, None, None)


class DeiTBlockFn(torch.autograd.Function):
    """Block_adapt.forward / Block.forward of TransFuse_S_adapt's DeiT branch (vision_transformer.py:172-211):
    x + attn(LN1(x)[, label]); then + mlp(LN2(.)).  LayerNorm kernels, bf16 tcgen05 GEMMs with the bias / GELU / residual
    epilogues, mdv_sdpa_fwd / mdv_sdpa_bwd.  drop = attn_drop = drop_path = 0 (the reference's DeiT-S setting)."""

    @staticmethod
    def forward(ctx, x, label, n1w, n1b, qkv_w, qkv_b, proj_w, proj_b, da_w1, da_b1, da_w2, da_b2, n2w, n2b, fc1_w, fc1_b, fc2_w, fc2_b,
                heads, scale, eps):
        B, N, C = x.shape
        M, dev = B * N, x.device
        hidden = fc1_w.shape[0]
        x = _contig(x.float())
        lib = L.lib()
        with _dev_ctx(x):
            ln1, mean1, rstd1 = layernorm_fwd(x, [n1w], [n1b], M, C, eps)
            qkv = torch.empty((M, 3 * C), dtype=BF16, device=dev)
            gemm_nt(ln1, prep_weight(qkv_w, 0, 3 * C, C), M, 3 * C, C, qkv, bias=qkv_b)
            gate = hid = None
            if da_w1 is not None:
                label = _contig(label.float())
                nd, hd = da_w1.shape[1], da_w1.shape[0]
                gate = torch.empty((B, C), dtype=F32, device=dev)
                hid = torch.empty((B, hd), dtype=F32, device=dev)
                check(lib.mdv_da_gate_fwd(ptr(label), ptr(da_w1), ptr(da_b1), ptr(da_w2), ptr(da_b2), ptr(hid), ptr(gate), B, nd, hd, C, heads,
                                          L.stream()), "mdv_da_gate_fwd")
            y = torch.empty((M, C), dtype=BF16, device=dev)
            lse = torch.empty((B, heads, N), dtype=F32, device=dev)
            check(lib.mdv_sdpa_fwd(ptr(qkv), ptr(gate), ptr(y), ptr(lse), B, N, C, heads, ctypes.c_float(scale), L.stream()), "mdv_sdpa_fwd")
            x2 = torch.empty((M, C), dtype=F32, device=dev)
            gemm_nt(y, prep_weight(proj_w, 0, C, C), M, C, C, x2, bias=proj_b, residual=x)
            ln2, mean2, rstd2 = layernorm_fwd(x2, [n2w], [n2b], M, C, eps)
            u = torch.empty((M, hidden), dtype=BF16, device=dev)
            hact = torch.empty((M, hidden), dtype=BF16, device=dev)
            gemm_nt(ln2, prep_weight(fc1_w, 0, hidden, C), M, hidden, C, hact, bias=fc1_b, act=ACT_GELU, out_preact=u, preact_mode=1)
            x3 = torch.empty((B, N, C), dtype=F32, device=dev)
            gemm_nt(hact, prep_weight(fc2_w, 0, C, hidden), M, C, hidden, x3, bias=fc2_b, residual=x2)
        ctx.save_for_backward(x, mean1, rstd1, ln1, qkv, y, lse, gate, hid, label if da_w1 is not None else None, x2, mean2, rstd2, ln2, u, hact)
        ctx.params = (n1w, n1b, qkv_w, qkv_b, proj_w, proj_b, da_w1, da_b1, da_w2, da_b2, n2w, n2b, fc1_w, fc1_b, fc2_w, fc2_b)
        ctx.meta = (B, N, C, hidden, heads, float(scale))
        _fwd_mark(ctx)
        return x3

    @staticmethod
    def backward(ctx, dx3):
        x, mean1, rstd1, ln1, qkv, y, lse, gate, hid, label, x2, mean2, rstd2, ln2, u, hact = ctx.saved_tensors
        names = ("n1w", "n1b", "qkv_w", "qkv_b", "proj_w", "proj_b", "da_w1", "da_b1", "da_w2", "da_b2", "n2w", "n2b", "fc1_w", "fc1_b",
                 "fc2_w", "fc2_b")
        P = dict(zip(names, ctx.params))
        B, N, C, hidden, heads, scale = ctx.meta
        M, dev = B * N, x.device
        lib = L.lib()
        dx3 = _contig(dx3.float())
        T = {n: gtarget(P[n], da=n.startswith("da_")) for n in names}
        G = {k: v[0] for k, v in T.items()}
        with _dev_ctx(x):
            d_fc2 = cast_bf16(dx3, M, C, colsum=G["fc2_b"])
            gemm_tn(d_fc2, hact, M, C, hidden, G["fc2_w"])
            du = torch.empty((M, hidden), dtype=BF16, device=dev)
            gemm_nt(d_fc2, prep_weight(P["fc2_w"], 1, C, hidden), M, hidden, C, du, mul_gelu_grad=u, mul_mode=1, colsum=G["fc1_b"])
            gemm_tn(du, ln2, M, hidden, C, G["fc1_w"])
            dln2 = torch.empty((M, C), dtype=F32, device=dev)
            gemm_nt(du, prep_weight(P["fc1_w"], 1, hidden, C), M, C, hidden, dln2)
            dx2, d_proj = layernorm_bwd(dln2, x2, mean2, rstd2, [P["n2w"]], dx3, M, C, [G["n2w"]], [G["n2b"]], masked=True,
                                        dbias_masked=G["proj_b"])
            gemm_tn(d_proj, y, M, C, C, G["proj_w"])
            dy = torch.empty((M, C), dtype=BF16, device=dev)
            gemm_nt(d_proj, prep_weight(P["proj_w"], 1, C, C), M, C, C, dy)
            dqkv = torch.empty((M, 3 * C), dtype=BF16, device=dev)
            dgate = torch.empty((B, C), dtype=F32, device=dev) if gate is not None else None
            check(lib.mdv_sdpa_bwd(ptr(qkv), ptr(gate), ptr(y), ptr(lse), ptr(dy), ptr(dqkv), ptr(dgate), B, N, C, heads, ctypes.c_float(scale),
                                   L.stream()), "mdv_sdpa_bwd")
            if gate is not None and G["da_w1"] is not None:
                nd, hd = P["da_w1"].shape[1], P["da_w1"].shape[0]
                ws2 = torch.empty(B * (C + hd), dtype=F32, device=dev)
                check(lib.mdv_da_gate_bwd(ptr(label), ptr(P["da_w2"]), ptr(hid), ptr(gate), ptr(dgate), ptr(G["da_w1"]), ptr(G["da_b1"]),
                                          ptr(G["da_w2"]), ptr(G["da_b2"]), ptr(ws2), B, nd, hd, C, heads, L.stream()), "mdv_da_gate_bwd")
            gemm_tn(dqkv, ln1, M, 3 * C, C, G["qkv_w"])
            colsum(dqkv, M, 3 * C, G["qkv_b"])
            dln1 = torch.empty((M, C), dtype=F32, device=dev)
            gemm_nt(dqkv, prep_weight(P["qkv_w"], 1, 3 * C, C), M, C, 3 * C, dln1)
            dx, _ = layernorm_bwd(dln1, x, mean1, rstd1, [P["n1w"]], dx2, M, C, [G["n1w"]], [G["n1b"]])
        _grads_done(ctx)
        return (dx.view(B, N, C), None, *[T[n][1] for n in names], None, None, None)


class DeiTEmbedFn(torch.autograd.Function):
    """PatchEmbed (Conv2d kernel = stride = patch: one GEMM over the flattened patches) + positional embedding
    (vision_transformer.py:214-236, DeiT.py:116-125).  `patches` [B*n, 3*p*p] are the image's patches in (c, i, j) order."""

    @staticmethod
    def forward(ctx, patches, w, b, pos, B, n):
        M, K = patches.shape
        C = w.shape[0]
        dev = patches.device
        with _dev_ctx(patches):
            pb = cast_bf16(_contig(patches.float()), M, K)
            pe = _contig(pos.reshape(1, n, C).expand(B, n, C)).view(M, C)
            out = torch.empty((B, n, C), dtype=F32, device=dev)
            gemm_nt(pb, prep_weight(w, 0, C, K), M, C, K, out, bias=b, residual=pe)
        ctx.save_for_backward(pb)
        ctx.params = (w, b, pos)
        ctx.meta = (B, n, C, K)
        _fwd_mark(ctx)
        return out

    @staticmethod
    def backward(ctx, dout):
        (pb,) = ctx.saved_tensors
        w, b, pos = ctx.params
        B, n, C, K = ctx.meta
        M = B * n
        dout = _contig(dout.float())
        with _dev_ctx(dout):
            g_w, r_w = gtarget(w, (C, K))
            gemm_tn(cast_bf16(dout, M, C), pb, M, C, K, g_w)
            g_b, r_b = gtarget(b)
            colsum(dout, M, C, g_b)
            g_p, r_p = gtarget(pos, (n * C,))
            colsum(dout, B, n * C, g_p)          # sum over the batch: rows = images
        _grads_done(ctx)
        return None, r_w, r_b, r_p, None, None


class LayerNormOutFn(torch.autograd.Function):
    """A LayerNorm whose output leaves the library (the final norm of the DeiT branch): fp32 in, fp32 out."""

    @staticmethod
    def forward(ctx, x, w, b, eps):
        B, N, C = x.shape
        x = _contig(x.float())
        with _dev_ctx(x):
            y, mean, rstd = layernorm_fwd(x, [w], [b], B * N, C, eps)
        ctx.save_for_backward(x, mean, rstd)
        ctx.params = (w, b)
        _fwd_mark(ctx)
        return y.float().view(B, N, C)

    @staticmethod
    def backward(ctx, dy):
        x, mean, rstd = ctx.saved_tensors
        w, b = ctx.params
        B, N, C = x.shape
        dy = _contig(dy.float())
        with _dev_ctx(x):
            g_w, r_w = gtarget(w)
            g_b, r_b = gtarget(b)
            dx, _ = layernorm_bwd(dy, x, mean, rstd, [w], None, B * N, C, [g_w], [g_b])
        _grads_done(ctx)
        return dx.view(B, N, C), r_w, r_b, None


class HeadFn(torch.autograd.Function):
    """bilinear up to the image size -> 1x1 conv C->1 (mdvit.py:699-700), evaluated as conv-then-resize (exact)."""

    @staticmethod
    def forward(ctx, x, w, b, H, W, Ho, Wo):
        B, _, C = x.shape
        dev = x.device
        x = _contig(x)
        lib = L.lib()
        with _dev_ctx(x):
            lo = torch.empty(B * H * W, dtype=F32, device=dev)
            check(lib.mdv_rowdot_fwd(ptr(x), 0, ptr(w), ptr(b), ptr(lo), B * H * W, C, H * W, ctypes.c_float(0.0), None, 0, L.stream()),
                  "mdv_rowdot_fwd")
            out = upsample_fwd(lo, torch.empty((B, 1, Ho, Wo), dtype=F32, device=dev), B, H, W, Ho, Wo, 1)
        ctx.save_for_backward(x)
        ctx.params = (w, b)
        ctx.meta = (B, C, H, W, Ho, Wo)
        _fwd_mark(ctx)
        return out

    @staticmethod
    def backward(ctx, dout):
        (x,) = ctx.saved_tensors
        w, b = ctx.params
        B, C, H, W, Ho, Wo = ctx.meta
        dev = x.device
        lib = L.lib()
        dout = _contig(dout.float())
        with _dev_ctx(x):
            dlo = upsample_bwd(dout, B, H, W, Ho, Wo, 1)
            dx = torch.empty((B, H * W, C), dtype=F32, device=dev)
            dw, rw = gtarget(w)
            db, rb = gtarget(b)
            check(lib.mdv_rowdot_bwd(ptr(dlo), ptr(x), 0, ptr(w), ptr(dx), ptr(dw), ptr(db), B * H * W, C, H * W, ctypes.c_float(0.0),
                                     None, 0, L.stream()), "mdv_rowdot_bwd")
        _grads_done(ctx)
        return dx, rw, rb, None, None, None, None


def _bf16_t(w, R, Cc):
    """bf16 [Cc, R] = w^T of a contiguous fp32 [R, Cc] that is not a parameter (no operand cache: recomputed every forward)."""
    dst = torch.empty((Cc, R), dtype=BF16, device=w.device)
    check(L.lib().mdv_prep_weight(ptr(w), ptr(dst), R, Cc, R, 1, 0, L.stream()), "mdv_prep_weight")
    return dst


class AuxFn(torch.autograd.Function):
    """MLPDecoderFM.forward (Decoders.py:315-339): the MKD auxiliary 'peer' decoder, with linear_fuse folded into linear1-4.

    A bilinear resize (align_corners=False) is linear per channel with weights summing to 1, and a 1x1 conv is linear per
    pixel, so with Wf_i the column block of linear_fuse's weight that multiplies input i (order x1..x4, x5):
        z = Wf . cat(up(W_i x_i + b_i), x5) + bf = [W'_1 | Wf_5] . [x1 | x5] + bf + c_1 + sum_{i=2..4} up(W'_i x_i + c_i),
        W'_i = Wf_i W_i,   c_i = Wf_i b_i.
    The [M0, 2112] concat and its K = 2112 GEMMs never exist: z is one K = C1 + C5 GEMM at full resolution, three GEMMs at
    the stage resolutions (outputs y_i kept in fp32) and one upsample-accumulate pass.  W'_i and c_i are computed in fp32
    from the master weights in every forward (so a captured step graph sees each optimizer update).  Backward, with dz the
    gradient of z, dz_i = up^T(dz) and s = colsum(dz) (= colsum(dz_i)):
        dx1 | dx5 = dz [W'_1 | Wf_5],  dx_i = dz_i W'_i,  E_i = dz_i^T x_i,
        dWf_i += E_i W_i^T + s b_i^T,  dWf_5 += E_5,  dW_i += Wf_i^T E_i,  db_i += Wf_i^T s,  dbf += s."""

    @staticmethod
    def forward(ctx, x1, x2, x3, x4, x5, l1w, l1b, l2w, l2b, l3w, l3b, l4w, l4b, fw, fb, g, b, ow, ob, bufs, sizes, Ho, Wo, drop2d,
                training):
        B = x1.shape[0]
        dev = x1.device
        xs = [_contig(t) for t in (x1, x2, x3, x4)]
        x5 = _contig(x5) if x5 is not None else None      # None: MLPDecoder (Decoders.py:239-286), no main-decoder feature
        (H, W) = sizes[0]
        M0 = B * H * W
        hc = fw.shape[0]               # 512
        K = fw.shape[1]                # 2112 (MLPDecoderFM) / 2048 (MLPDecoder)
        C5 = x5.shape[2] if x5 is not None else 0
        Cs = [t.shape[2] for t in xs]
        C1 = Cs[0]
        Kx = C1 + C5
        rm, rv, nb = bufs
        lib = L.lib()
        lw, lb = (l1w, l2w, l3w, l4w), (l1b, l2b, l3b, l4b)
        with _dev_ctx(x1):
            # collapsed weights: w1x = [W'_1 | Wf_5] (fp32 [hc, Kx]) and W'_2..4; bias c_i = Wf_i b_i (c_1 also takes bf), added to
            # the stage-i product before the resize (a resize keeps constants)
            w1x = torch.empty((hc, Kx), dtype=F32, device=dev)
            if C5:
                check(lib.mdv_add_f32(ptr(fw[:, 4 * hc:]), 0, K, ptr(w1x[:, C1:]), Kx, hc, C5, 0, L.stream()), "mdv_add_f32")
            wps = [torch.empty((hc, Cs[i]), dtype=F32, device=dev) for i in range(1, 4)]
            cb = torch.empty((4, hc), dtype=F32, device=dev)
            check(lib.mdv_add_f32(ptr(fb), 0, hc, ptr(cb), hc, 1, hc, 0, L.stream()), "mdv_add_f32")
            matmul_f32([mm(fw, lw[0], w1x, hc, C1, hc, lda=K, ldc=Kx)] +
                       [mm(fw[:, i * hc:], lw[i], wps[i - 1], hc, Cs[i], hc, lda=K) for i in range(1, 4)] +
                       [mm(fw[:, i * hc:], lb[i], cb[i], hc, 1, hc, lda=K, accumulate=i == 0) for i in range(4)])
            # z = [x1 | x5] . w1x^T + c_1 + sum_i up(x_i . W'_i^T + c_i)
            xa = torch.empty((M0, Kx), dtype=BF16, device=dev)
            cast_bf16(xs[0], M0, C1, out=xa, ld_out=Kx)
            if C5:
                cast_bf16(x5, M0, C5, out=xa[:, C1:], ld_out=Kx)
            z = torch.empty((M0, hc), dtype=F32, device=dev)
            gemm_nt(xa, cast_bf16(w1x, hc, Kx), M0, hc, Kx, z, bias=cb[0])
            acts, ys = [xa], []
            for i in range(1, 4):
                Hi, Wi = sizes[i]
                Mi, Ci = B * Hi * Wi, Cs[i]
                a = cast_bf16(xs[i], Mi, Ci)
                acts.append(a)
                ys.append((gemm_nt(a, cast_bf16(wps[i - 1], hc, Ci), Mi, hc, Ci, torch.empty((Mi, hc), dtype=F32, device=dev), bias=cb[i]), Hi, Wi))
            upsample_add(z, ys, B, H, W, hc)
            a5, mean, rstd = bn_forward(z, M0, hc, [g], [b], [rm], [rv], [nb], training, ACT_RELU, True)
            p2 = drop2d if training else 0.0
            sid = new_stream_id() if p2 > 0 else 0
            lo = torch.empty(M0, dtype=F32, device=dev)
            check(lib.mdv_rowdot_fwd(ptr(a5), 1, ptr(ow), ptr(ob), ptr(lo), M0, hc, H * W, ctypes.c_float(p2),
                                     ptr(rng_tensor(dev)) if p2 > 0 else None, sid, L.stream()), "mdv_rowdot_fwd")
            out = upsample_fwd(lo, torch.empty((B, 1, Ho, Wo), dtype=F32, device=dev), B, H, W, Ho, Wo, 1)
            if training:     # input-gradient operands: bf16 transposes of the collapsed weights
                wts = [_bf16_t(w1x, hc, Kx)] + [_bf16_t(wps[i - 1], hc, Cs[i]) for i in range(1, 4)]
            else:
                wts, z = [], None
        ctx.save_for_backward(z, mean, rstd, a5, *acts, *wts)
        ctx.params = (l1w, l1b, l2w, l2b, l3w, l3b, l4w, l4b, fw, fb, g, b, ow, ob)
        ctx.meta = (B, sizes, Ho, Wo, hc, K, C5, p2, sid, training, Cs)
        _fwd_mark(ctx)
        return out

    @staticmethod
    def backward(ctx, dout):
        B, sizes, Ho, Wo, hc, K, C5, p2, sid, training, Cs = ctx.meta
        _require_train_bn(training)
        z, mean, rstd, a5, *rest = ctx.saved_tensors
        acts, wts = rest[:4], rest[4:]
        l1w, l1b, l2w, l2b, l3w, l3b, l4w, l4b, fw, fb, g, b, ow, ob = ctx.params
        (H, W) = sizes[0]
        M0, dev = B * H * W, dout.device
        C1 = Cs[0]
        Kx = C1 + C5
        lib = L.lib()
        dout = _contig(dout.float())
        lw, lb = (l1w, l2w, l3w, l4w), (l1b, l2b, l3b, l4b)
        with _dev_ctx(dout):
            dlo = upsample_bwd(dout, B, H, W, Ho, Wo, 1)
            g_ow, r_ow = gtarget(ow)
            g_ob, r_ob = gtarget(ob)
            if g_ow is not None:    # weight / bias gradient of linear_out only: d(a5) is never materialised (rank-1, see below)
                check(lib.mdv_rowdot_bwd(ptr(dlo), ptr(a5), 1, ptr(ow), None, ptr(g_ow), ptr(g_ob), M0, hc, H * W, ctypes.c_float(p2),
                                         ptr(rng_tensor(dev)) if p2 > 0 else None, sid, L.stream()), "mdv_rowdot_bwd")
            # BatchNorm backward with d(a5)[m,c] = dlo[m] * w_out[c] * dropout2d_mask generated on the fly
            dz = torch.empty((M0, hc), dtype=BF16, device=dev)
            ws_bn = torch.empty(3 * hc + (B * hc + 1) // 2, dtype=torch.float64, device=dev)
            g_g, rg = gtarget(g)
            g_b, rb = gtarget(b)
            check(lib.mdv_bn_act_bwd_rank1(ptr(dlo), ptr(ow), H * W, ctypes.c_float(p2), ptr(rng_tensor(dev)) if p2 > 0 else None, sid,
                                           ptr(z), ptr(mean), ptr(rstd), ptr(g), ptr(b), ACT_RELU, ptr(dz), 1, ptr(g_g), ptr(g_b), M0, hc,
                                           ptr(ws_bn), L.stream()), "mdv_bn_act_bwd_rank1")
            g_fw, r_fw = gtarget(fw, (hc, K))
            g_fb, r_fb = gtarget(fb)
            tw = [gtarget(lw[i], (hc, Cs[i])) for i in range(4)]
            tb = [gtarget(lb[i]) for i in range(4)]
            wgrad = any(t is not None for t in [g_fw, g_fb] + [t[0] for t in tw + tb])
            gx = [gemm_nt(dz, wts[0], M0, C1, hc, torch.empty((B, H * W, C1), dtype=F32, device=dev))]
            dx5 = gemm_nt(dz, wts[0][C1:], M0, C5, hc, torch.empty((B, H * W, C5), dtype=F32, device=dev)) if C5 else None
            if wgrad:
                s = colsum(dz, M0, hc, torch.zeros(hc, dtype=F32, device=dev))
                Es = [gemm_tn(dz, acts[0], M0, hc, Kx, torch.zeros((hc, Kx), dtype=F32, device=dev))]
            for i in range(1, 4):
                Hi, Wi = sizes[i]
                Mi, Ci = B * Hi * Wi, Cs[i]
                dzi = cast_bf16(upsample_bwd(dz, B, Hi, Wi, H, W, hc), Mi, hc)
                gx.append(gemm_nt(dzi, wts[i], Mi, Ci, hc, torch.empty((B, Hi * Wi, Ci), dtype=F32, device=dev)))
                if wgrad:
                    Es.append(gemm_tn(dzi, acts[i], Mi, hc, Ci, torch.zeros((hc, Ci), dtype=F32, device=dev)))
            if wgrad:
                probs = []
                for i in range(4):
                    Ci, ldE = Cs[i], (Kx if i == 0 else Cs[i])
                    wf = fw[:, i * hc:]
                    gwf = g_fw[:, i * hc:] if g_fw is not None else None
                    probs += [mm(Es[i], lw[i], gwf, hc, hc, Ci, lda=ldE, ldc=K, trans_b=True, accumulate=True, u=s, v=lb[i]),
                              mm(wf, Es[i], tw[i][0], hc, Ci, hc, lda=K, ldb=ldE, trans_a=True, accumulate=True),
                              mm(wf, s, tb[i][0], hc, 1, hc, lda=K, trans_a=True, accumulate=True)]
                matmul_f32(probs)
                if g_fw is not None and C5:
                    check(lib.mdv_add_f32(ptr(Es[0][:, C1:]), 0, Kx, ptr(g_fw[:, 4 * hc:]), K, hc, C5, 1, L.stream()), "mdv_add_f32")
                if g_fb is not None:
                    check(lib.mdv_add_f32(ptr(s), 0, hc, ptr(g_fb), hc, 1, hc, 1, L.stream()), "mdv_add_f32")
        _grads_done(ctx)
        return (gx[0], gx[1], gx[2], gx[3], dx5, tw[0][1], tb[0][1], tw[1][1], tb[1][1], tw[2][1], tb[2][1], tw[3][1], tb[3][1], r_fw,
                r_fb, rg, rb, r_ow, r_ob, None, None, None, None, None, None)


# ------------------------------------------------------------------------------------------------- domain split
class SplitDomainsFn(torch.autograd.Function):
    """x [G*B, ...] -> G views [B, ...] (the per-domain slices the auxiliary decoders consume in MDViT.forward_multi).
    Plain slicing would make autograd zero-fill and add a full-size tensor per slice in backward; here the G slice
    gradients are concatenated once."""

    @staticmethod
    def forward(ctx, x, G):
        B = x.shape[0] // G
        ctx.G, ctx.shape_b = G, (B,) + tuple(x.shape[1:])
        return tuple(x.narrow(0, g * B, B) for g in range(G))

    @staticmethod
    def backward(ctx, *grads):
        ref = next(g for g in grads if g is not None)
        parts = [g if g is not None else torch.zeros(ctx.shape_b, dtype=ref.dtype, device=ref.device) for g in grads]
        return torch.cat(parts, dim=0), None


# ------------------------------------------------------------------------------------------------- fused losses
def _label_arg(label):
    """Labels as the trainer hands them over: fp32 (label.cuda().float(), multi_train_MDViT.py:136) or uint8 {0,1}."""
    if label.dtype == torch.uint8:
        return _contig(label), 1
    return _contig(label.float()), 0


class SegLossFn(torch.autograd.Function):
    """(L_seg, L_aux, L_kt) of multi_train_MDViT.py:147-169 for G domain mini-batches at once: one pass over each
    (out, aux, label) -> [G,8] partial sums; `reduce_sums` (optional callable) all-reduces them ONCE across data-parallel
    ranks so BCE/Dice are those of the gathered global batch; -> losses [G,3].  Inputs: out_0.., aux_0.. (or None), label_0.."""

    @staticmethod
    def forward(ctx, n_total, reduce_sums, G, *tensors):
        outs = [_contig(t.float()) for t in tensors[:G]]
        auxs = [(_contig(t.float()) if t is not None else None) for t in tensors[G:2 * G]]
        labs = [_label_arg(t) for t in tensors[2 * G:3 * G]]
        dev = outs[0].device
        lib = L.lib()
        with _dev_ctx(outs[0]):
            sums = torch.empty((G, 8), dtype=torch.float64, device=dev)
            for g in range(G):
                check(lib.mdv_loss_sums(ptr(outs[g]), ptr(auxs[g]), ptr(labs[g][0]), labs[g][1], ptr(sums[g]), outs[g].numel(), L.stream()),
                      "mdv_loss_sums")
            if reduce_sums is not None:
                reduce_sums(sums)
            losses = torch.empty((G, 3), dtype=F32, device=dev)
            nt = [float(n_total or o.numel()) for o in outs]
            for g in range(G):
                check(lib.mdv_loss_finalize(ptr(sums[g]), ctypes.c_double(nt[g]), ptr(losses[g]), L.stream()), "mdv_loss_finalize")
        ctx.save_for_backward(sums, *outs, *[a for a in auxs if a is not None], *[l for l, _ in labs])
        ctx.G, ctx.nt, ctx.has_aux, ctx.lab_u8 = G, nt, [a is not None for a in auxs], [u for _, u in labs]
        return losses

    @staticmethod
    def backward(ctx, dl):
        G = ctx.G
        sums, *rest = ctx.saved_tensors
        outs, rest = rest[:G], rest[G:]
        na = sum(ctx.has_aux)
        it = iter(rest[:na])
        auxs = [next(it) if h else None for h in ctx.has_aux]
        labs = rest[na:]
        lib = L.lib()
        dl = _contig(dl.float())
        douts, dauxs = [], []
        with _dev_ctx(outs[0]):
            for g in range(G):
                dout = torch.empty_like(outs[g])
                daux = torch.empty_like(auxs[g]) if auxs[g] is not None else None
                check(lib.mdv_loss_bwd(ptr(outs[g]), ptr(auxs[g]), ptr(labs[g]), ctx.lab_u8[g], ptr(sums[g]), ctypes.c_double(ctx.nt[g]),
                                       ptr(dl[g]), ptr(dout), ptr(daux), outs[g].numel(), L.stream()), "mdv_loss_bwd")
                douts.append(dout)
                dauxs.append(daux)
        return (None, None, None, *douts, *dauxs, *([None] * G))


def seg_losses_multi(outs, auxs, labels, n_total=None, reduce_sums=None):
    """[G,3] losses (seg, aux, kt) of G domain mini-batches; one all-reduce of the [G,8] partial sums when data-parallel."""
    G = len(outs)
    return SegLossFn.apply(n_total, reduce_sums, G, *outs, *auxs, *labels)


def seg_losses(out, aux, label, n_total=None, reduce_sums=None):
    return seg_losses_multi([out], [aux], [label], n_total, reduce_sums)[0]


def seg_counts(logits, label, counts=None):
    """Device-side Dice/Jaccard counts {|P&L|, |P|, |L|} (int64[3], accumulated) of the thresholded prediction — replaces the
    per-domain `output.cpu().numpy()` + medpy dc/jc host round trip of multi_train_MDViT.py:172-177; read back when logging."""
    logits = _contig(logits.detach().float())
    lab, u8 = _label_arg(label)
    if counts is None:
        counts = torch.zeros(3, dtype=torch.int64, device=logits.device)
    with _dev_ctx(logits):
        check(L.lib().mdv_seg_counts(ptr(logits), ptr(lab), u8, ptr(counts), logits.numel(), L.stream()), "mdv_seg_counts")
    return counts


def dice_jaccard(counts):
    """(dc, jc) from seg_counts() with medpy.metric.binary semantics (0.0 when the denominator is empty)."""
    c = counts.tolist()
    dc = 2.0 * c[0] / (c[1] + c[2]) if (c[1] + c[2]) > 0 else 0.0
    jc = c[0] / (c[1] + c[2] - c[0]) if (c[1] + c[2] - c[0]) > 0 else 0.0
    return dc, jc


# ------------------------------------------------------------------------------------------------- TransFuse_S_adapt: CNN side
# Dense convolutions of the ResNet34 branch, BiFusion blocks, Up blocks and output heads
# (Models/Hybrid_models/TransFuseFolder/TransFuse.py:182-283, 556-650; torchvision resnet34 BasicBlock) on NHWC fp32 maps
# ([B, H*W, C]): im2col + TF32 tcgen05 GEMM forward, bf16 tcgen05 GEMMs for the input / weight gradients.
def conv_geom(H, W, k, stride):
    pad = (k - 1) // 2
    return (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1, pad


_IMPLICIT_CONV = not bool(int(_os.environ.get("MDV_NO_IMPLICIT_CONV", "0")))      # A/B switch (development)


def implicit_conv_ok(H, W, Cin, bf16):
    """mdv_conv3_gemm's geometry: 128-row tiles are whole image rows, channel chunks fill a 128-byte k-block"""
    return _IMPLICIT_CONV and W <= 128 and 128 % W == 0 and (H * W) % 128 == 0 and Cin % (64 if bf16 else 32) == 0


def conv3_gemm(x, Wm, B, H, W, Cin, N, out, *, flip=False, bias=None):
    """out [B*H*W, N] = 3x3/stride-1/pad-1 convolution of the NHWC map x as one implicit tcgen05 GEMM (mdv_conv3_gemm)"""
    e = GemmEpi()
    e.bias, e.out, e.ldc = ptr(bias), ptr(out), N
    e.out_bf16 = 1 if out.dtype == BF16 else 0
    e.rows_per_scale = 1
    check(L.lib().mdv_conv3_gemm(ptr(x), int(x.dtype == F32), Cin, ptr(Wm), Wm.shape[1], B, H, W, Cin, N, int(flip), ctypes.byref(e),
                                 L.stream()), "mdv_conv3_gemm")
    return out


def _conv_cols(x, B, H, W, Cin, k, stride, nchw, Cout=0):
    """fp32 A operand of the conv GEMM: (A [M, ld], ld, kind).  kind 'direct': the map itself (1x1, stride 1); 'k3i': the map
    itself, read by the implicit-GEMM kernel (3x3, stride 1; no im2col matrix); 'k3': im2col in (tap, channel) order
    (mdv_im2col3); 'gen': generic k x k im2col in the flattened-weight (channel, tap) order."""
    Ho, Wo, pad = conv_geom(H, W, k, stride)
    M, dev = B * Ho * Wo, x.device
    lib = L.lib()
    if k == 1 and stride == 1 and not nchw and Cin % 8 == 0:
        return x.view(M, Cin), Cin, "direct"
    if k == 3 and stride == 1 and not nchw and Cout > 1 and Cin % 8 == 0 and implicit_conv_ok(H, W, Cin, False):
        return x.view(M, Cin), 9 * Cin, "k3i"
    if k == 3 and not nchw and Cin % 8 == 0:
        col = torch.empty((M, 9 * Cin), dtype=F32, device=dev)
        check(lib.mdv_im2col3(ptr(x), 0, ptr(col), 0, B, H, W, Ho, Wo, Cin, stride, 9 * Cin, L.stream()), "mdv_im2col3")
        return col, 9 * Cin, "k3"
    K = Cin * k * k
    ld = (K + 7) // 8 * 8
    col = torch.empty((M, ld), dtype=F32, device=dev)
    check(lib.mdv_im2col_k(ptr(x), int(nchw), ptr(col), 0, B, H, W, Ho, Wo, Cin, k, stride, pad, ld, L.stream()), "mdv_im2col_k")
    return col, ld, "gen"


def _conv_weight_f32(w, kind, ld):
    """fp32 W operand [Cout, ld] matching _conv_cols' column order."""
    Cout, Cin, k = w.shape[0], w.shape[1], w.shape[2]
    if kind in ("k3", "k3i"):
        return prep_weight(w, 2 | 8, Cout, 9 * Cin, cin=Cin)
    K = Cin * k * k
    if ld == K:
        return _contig(w).view(Cout, K)
    dst = torch.zeros((Cout, ld), dtype=F32, device=w.device)
    with torch.no_grad():
        check(L.lib().mdv_prep_weight(ptr(_contig(w)), ptr(dst), Cout, K, ld, 0 | 8, 0, L.stream()), "mdv_prep_weight")
    return dst


class ConvBnActFn(torch.autograd.Function):
    """y = act( BN?( conv_kxk(x) + bias? ) + residual? ) on NHWC maps: nn.Conv2d (+ nn.BatchNorm2d) (+ `out += identity`) (+ ReLU)
    of TransFuse.py's Conv / DoubleConv / Residual / Attention_block and of torchvision's BasicBlock.  k in {1,3,7}, stride in
    {1,2}, padding (k-1)//2.  x: [B, H*W, Cin] fp32, or the NCHW image [B, Cin, H, W] (nchw=True, resnet.conv1).  Cout == 1
    (the output heads and BiFusion_block.spatial) runs as a row dot product instead of a GEMM (no BN / residual there)."""

    @staticmethod
    def forward(ctx, x, w, cbias, gamma, beta, residual, bufs, B, H, W, stride, act, training, nchw):
        if not x.is_cuda:
            raise RuntimeError("mdvit_b200 runs on CUDA (sm_100a) only; there is no CPU path")
        Cout, Cin, k = w.shape[0], w.shape[1], w.shape[2]
        Ho, Wo, pad = conv_geom(H, W, k, stride)
        M, dev = B * Ho * Wo, x.device
        x = _contig(x)
        has_bn = gamma is not None
        lib = L.lib()
        with _dev_ctx(x):
            A, ld, kind = _conv_cols(x, B, H, W, Cin, k, stride, nchw, Cout)
            Wf = _conv_weight_f32(w, kind, ld)
            z = mean = rstd = None

            def conv_out(**kw):      # fp32 [M, Cout] = conv(x) (+ bias ...)
                o = torch.empty((M, Cout), dtype=F32, device=dev)
                if kind == "k3i":
                    return conv3_gemm(A, Wf, B, H, W, Cin, Cout, o, bias=kw.get("bias"))
                return gemm_nt(A, Wf, M, Cout, ld, o, tf32=True, **kw)

            if Cout == 1:
                if has_bn or residual is not None or act != ACT_NONE:
                    raise NotImplementedError("single-channel conv: no BN / residual / activation")
                y = torch.empty(M, dtype=F32, device=dev)
                check(lib.mdv_rowdot_fwd(ptr(A), 0, ptr(Wf), ptr(cbias), ptr(y), M, ld, Ho * Wo, ctypes.c_float(0.0), None, 0, L.stream()),
                      "mdv_rowdot_fwd")
            elif not has_bn:
                if act != ACT_NONE and residual is not None:
                    raise NotImplementedError("activation after a residual add needs BN in between")
                res = _contig(residual).view(M, Cout) if residual is not None else None
                if kind == "k3i":
                    raise NotImplementedError("3x3 conv without BatchNorm (not part of TransFuse_S_adapt apart from the 1-channel heads)")
                y = gemm_nt(A, Wf, M, Cout, ld, torch.empty((M, Cout), dtype=F32, device=dev), bias=cbias, residual=res, act=act, tf32=True)
            else:
                rm, rv, nb = bufs
                z = conv_out(bias=cbias)
                if residual is None:
                    y, mean, rstd = bn_forward(z, M, Cout, [gamma], [beta], [rm], [rv], [nb], training, act, False)
                else:
                    t, mean, rstd = bn_forward(z, M, Cout, [gamma], [beta], [rm], [rv], [nb], training, ACT_NONE, False)
                    y = torch.empty((M, Cout), dtype=F32, device=dev)
                    check(lib.mdv_add_act(ptr(t), ptr(_contig(residual)), ptr(y), M * Cout, act, L.stream()), "mdv_add_act")
        need_y = act == ACT_RELU and (residual is not None or not has_bn)
        ctx.save_for_backward(A, z, mean, rstd, y if need_y else None)
        ctx.params = (w, cbias, gamma, beta)
        ctx.meta = (B, H, W, Ho, Wo, Cin, Cout, k, stride, pad, ld, kind, act, training, residual is not None, has_bn)
        _fwd_mark(ctx)
        return y.view(B, Ho * Wo, Cout)

    @staticmethod
    def backward(ctx, dy):
        B, H, W, Ho, Wo, Cin, Cout, k, stride, pad, ld, kind, act, training, has_res, has_bn = ctx.meta
        if has_bn:
            _require_train_bn(training)
        A, z, mean, rstd, y = ctx.saved_tensors
        w, cbias, gamma, beta = ctx.params
        M, dev = B * Ho * Wo, dy.device
        K = Cin * k * k
        lib = L.lib()
        dy = _contig(dy.float())
        rg = rb = dres = dx = None
        need_dx = ctx.needs_input_grad[0]
        with _dev_ctx(dy):
            if Cout == 1:
                gwv = torch.zeros(ld, dtype=F32, device=dev)
                gb, rcb = gtarget(cbias)
                dcol = torch.empty((M, ld), dtype=F32, device=dev) if need_dx else None
                Wf = _conv_weight_f32(w, kind, ld)
                check(lib.mdv_rowdot_bwd(ptr(dy), ptr(A), 0, ptr(Wf), ptr(dcol), ptr(gwv), ptr(gb), M, ld, Ho * Wo, ctypes.c_float(0.0), None, 0,
                                         L.stream()), "mdv_rowdot_bwd")
                gw, rw = gtarget(w)
                if gw is not None:
                    if kind == "k3":
                        check(lib.mdv_unperm_conv_grad(ptr(gwv), ld, ptr(gw), 1, Cin, L.stream()), "mdv_unperm_conv_grad")
                    else:
                        check(lib.mdv_add_f32(ptr(gwv), 0, ld, ptr(gw), K, 1, K, 1, L.stream()), "mdv_add_f32")
            else:
                g = dy.view(M, Cout)
                if y is not None:      # ReLU whose input is not the BatchNorm output alone: mask from the saved output
                    g = torch.empty((M, Cout), dtype=F32, device=dev)
                    check(lib.mdv_relu_bwd(ptr(dy), ptr(y), ptr(g), M * Cout, L.stream()), "mdv_relu_bwd")
                if has_res:
                    dres = g.view(B, Ho * Wo, Cout)
                if has_bn:
                    dz, (rg,), (rb,) = bn_backward(g, z, mean, rstd, [gamma], [beta], ACT_NONE if has_res else act, M, Cout)
                else:
                    dz = cast_bf16(g, M, Cout)
                gb, rcb = gtarget(cbias)
                colsum(dz, M, Cout, gb)
                implicit_wgrad = kind == "k3i" and _IMPLICIT_CONV and Cin % 64 == 0 and W <= 64 and 64 % W == 0 and (H * W) % 64 == 0
                if kind == "k3":
                    rw = _conv3_wgrad(dz, A, w)
                elif kind == "k3i" and not implicit_wgrad:
                    Ab = None
                    if wgrad_on():      # the im2col matrix exists only here, in bf16, as the weight-gradient GEMM's operand
                        Ab = torch.empty((M, ld), dtype=BF16, device=dev)
                        check(lib.mdv_im2col3(ptr(A), 0, ptr(Ab), 1, B, H, W, Ho, Wo, Cin, 1, ld, L.stream()), "mdv_im2col3")
                    rw = _conv3_wgrad(dz, Ab, w)
                else:
                    gw, rw = gtarget(w)
                    if gw is None:
                        pass
                    elif kind == "k3i":
                        # implicit weight-gradient GEMM: B tiles straight from a bf16 copy of the map
                        gwp = torch.zeros((Cout, ld), dtype=F32, device=dev)
                        check(lib.mdv_conv3_wgrad(ptr(dz), Cout, ptr(cast_bf16(A, M, Cin)), Cin, B, H, W, Cin, Cout, ptr(gwp), ld, L.stream()),
                              "mdv_conv3_wgrad")
                        check(lib.mdv_unperm_conv_grad(ptr(gwp), ld, ptr(gw), Cout, Cin, L.stream()), "mdv_unperm_conv_grad")
                    elif ld == K:
                        gemm_tn(dz, cast_bf16(A, M, ld), M, Cout, K, gw.view(Cout, K))
                    else:
                        gwp = gemm_tn(dz, cast_bf16(A, M, ld), M, Cout, ld, torch.zeros((Cout, ld), dtype=F32, device=dev))
                        check(lib.mdv_add_f32(ptr(gwp), 0, ld, ptr(gw), K, Cout, K, 1, L.stream()), "mdv_add_f32")
                dcol = None
                if need_dx:
                    if kind == "direct":
                        dx = gemm_nt(dz, prep_weight(w, 1, Cout, Cin), M, Cin, Cout, torch.empty((M, Cin), dtype=F32, device=dev))
                    elif kind == "k3i" and implicit_conv_ok(H, W, Cout, True):
                        # input gradient = the same implicit GEMM over dz with the taps mirrored: dx never exists as a [M, 9 Cin] matrix
                        dx = conv3_gemm(dz, prep_weight(w, 4, Cout, 9 * Cin), B, H, W, Cout, Cin, torch.empty((M, Cin), dtype=F32, device=dev),
                                        flip=True)
                    elif kind in ("k3", "k3i"):
                        dcol = gemm_nt(dz, prep_weight(w, 3, Cout, 9 * Cin, cin=Cin), M, 9 * Cin, Cout, torch.empty((M, ld), dtype=F32, device=dev))
                    else:
                        if K != ld:
                            raise NotImplementedError("input gradient of a generic conv needs Cin*k*k % 8 == 0")
                        dcol = gemm_nt(dz, prep_weight(w, 1, Cout, K), M, K, Cout, torch.empty((M, ld), dtype=F32, device=dev))
            if need_dx and dx is None and kind == "direct":
                dx = dcol
            elif need_dx and dx is None:
                dx = torch.empty((B * H * W, Cin), dtype=F32, device=dev)
                if kind in ("k3", "k3i"):
                    check(lib.mdv_col2im3(ptr(dcol), ptr(dx), B, H, W, Ho, Wo, Cin, stride, ld, L.stream()), "mdv_col2im3")
                else:
                    check(lib.mdv_col2im_k(ptr(dcol), ptr(dx), B, H, W, Ho, Wo, Cin, k, stride, pad, ld, L.stream()), "mdv_col2im_k")
        _grads_done(ctx)
        return (dx.view(B, H * W, Cin) if dx is not None else None, rw, rcb, rg, rb, dres, None, None, None, None, None, None, None, None)


class BnActFn(torch.autograd.Function):
    """y = act(BatchNorm2d(x)) on an NHWC map (the pre-activation BatchNorms of TransFuse.py's Residual block, :626-640)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, bufs, act, training):
        B, N, C = x.shape
        x = _contig(x)
        rm, rv, nb = bufs
        with _dev_ctx(x):
            y, mean, rstd = bn_forward(x.view(B * N, C), B * N, C, [gamma], [beta], [rm], [rv], [nb], training, act, False)
        ctx.save_for_backward(x, mean, rstd)
        ctx.params = (gamma, beta)
        ctx.meta = (B, N, C, act, training)
        _fwd_mark(ctx)
        return y.view(B, N, C)

    @staticmethod
    def backward(ctx, dy):
        B, N, C, act, training = ctx.meta
        _require_train_bn(training)
        x, mean, rstd = ctx.saved_tensors
        gamma, beta = ctx.params
        dy = _contig(dy.float())
        with _dev_ctx(dy):
            dx, (rg,), (rb,) = bn_backward(dy, x, mean, rstd, [gamma], [beta], act, B * N, C, dz_bf16=False)
        _grads_done(ctx)
        return dx.view(B, N, C), rg, rb, None, None, None


class MaxPool3s2Fn(torch.autograd.Function):
    """nn.MaxPool2d(kernel_size=3, stride=2, padding=1) of torchvision's resnet34 (TransFuse.py:234) on an NHWC map."""

    @staticmethod
    def forward(ctx, x, H, W):
        B, _, C = x.shape
        x = _contig(x)
        Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
        out = torch.empty((B, Ho * Wo, C), dtype=F32, device=x.device)
        tap = torch.empty((B, Ho * Wo, C), dtype=torch.uint8, device=x.device)
        with _dev_ctx(x):
            check(L.lib().mdv_maxpool3s2_fwd(ptr(x), ptr(out), ptr(tap), B, H, W, C, L.stream()), "mdv_maxpool3s2_fwd")
        ctx.save_for_backward(tap)
        ctx.meta = (B, H, W, C)
        return out

    @staticmethod
    def backward(ctx, dout):
        (tap,) = ctx.saved_tensors
        B, H, W, C = ctx.meta
        dout = _contig(dout.float())
        din = torch.empty((B, H * W, C), dtype=F32, device=dout.device)
        with _dev_ctx(dout):
            check(L.lib().mdv_maxpool3s2_bwd(ptr(dout), ptr(tap), ptr(din), B, H, W, C, L.stream()), "mdv_maxpool3s2_bwd")
        return din, None, None


class ResizeACFn(torch.autograd.Function):
    """Bilinear resize with align_corners=True on an NHWC map (nn.Upsample in Up, TransFuse.py:559; F.interpolate of the three
    output maps, TransFuse.py:262-264)."""

    @staticmethod
    def forward(ctx, x, H, W, Ho, Wo):
        B, _, C = x.shape
        x = _contig(x)
        out = torch.empty((B, Ho * Wo, C), dtype=F32, device=x.device)
        with _dev_ctx(x):
            check(L.lib().mdv_resize_ac_fwd(ptr(x), ptr(out), B, H, W, Ho, Wo, C, L.stream()), "mdv_resize_ac_fwd")
        ctx.meta = (B, H, W, Ho, Wo, C)
        return out

    @staticmethod
    def backward(ctx, dout):
        B, H, W, Ho, Wo, C = ctx.meta
        dout = _contig(dout.float())
        din = torch.empty((B, H * W, C), dtype=F32, device=dout.device)
        with _dev_ctx(dout):
            check(L.lib().mdv_resize_ac_bwd(ptr(dout), ptr(din), B, H, W, Ho, Wo, C, L.stream()), "mdv_resize_ac_bwd")
        return din, None, None, None, None


def structure_weit(mask):
    """weit = 1 + 5 |avg_pool2d(mask, 31, stride 1, padding 15) - mask| (multi_train_TransFuse.py:30); mask [B,1,H,W] fp32."""
    B, _, H, W = mask.shape
    mask = _contig(mask.float())
    weit, ws = torch.empty_like(mask), torch.empty_like(mask)
    with _dev_ctx(mask):
        check(L.lib().mdv_structure_weit(ptr(mask), ptr(weit), ptr(ws), B, H, W, L.stream()), "mdv_structure_weit")
    return weit


class StructureLossFn(torch.autograd.Function):
    """structure_loss(pred, mask) of multi_train_TransFuse.py:29-38 (weighted BCE + weighted IoU, mean over the batch)."""

    @staticmethod
    def forward(ctx, pred, mask, weit):
        B, HW = pred.shape[0], pred[0].numel()
        pred, mask = _contig(pred), _contig(mask.float())
        sums = torch.empty(4 * B, dtype=torch.float64, device=pred.device)
        loss = torch.empty(1, dtype=F32, device=pred.device)
        with _dev_ctx(pred):
            check(L.lib().mdv_structure_loss_fwd(ptr(pred), ptr(mask), ptr(weit), ptr(sums), ptr(loss), B, HW, L.stream()), "mdv_structure_loss_fwd")
        ctx.save_for_backward(pred, mask, weit, sums)
        s = sums.view(B, 4)
        per_sample = (s[:, 1] / s[:, 0] + 1.0 - (s[:, 2] + 1.0) / (s[:, 3] - s[:, 2] + 1.0)).float()
        ctx.mark_non_differentiable(per_sample)
        return loss[0], per_sample

    @staticmethod
    def backward(ctx, g, _unused=None):
        pred, mask, weit, sums = ctx.saved_tensors
        B, HW = pred.shape[0], pred[0].numel()
        g = _contig(g.float()).view(1)
        dpred = torch.empty_like(pred)
        with _dev_ctx(pred):
            check(L.lib().mdv_structure_loss_bwd(ptr(pred), ptr(mask), ptr(weit), ptr(sums), ptr(g), ctypes.c_float(1.0), ptr(dpred), B, HW, 0,
                                                 L.stream()), "mdv_structure_loss_bwd")
        return dpred, None, None


def structure_loss(pred, mask, weit=None, per_sample=False):
    """Drop-in for multi_train_TransFuse.py:29-38; pass `weit` (structure_weit(mask)) to share it between the three maps.
    per_sample=True also returns the [B] per-sample terms (wbce + wiou, detached) whose mean the loss is."""
    if weit is None:
        weit = structure_weit(mask)
    loss, ps = StructureLossFn.apply(pred, mask, weit)
    return (loss, ps) if per_sample else loss


class GateCatFn(torch.autograd.Function):
    """[ g * p | x * v | bp ] in one pass: the spatial / channel gates of BiFusion_block and the concat feeding its Residual block
    (TransFuse.py:63-73); with x = v = bp = None, Attention_block's `x * psi` (TransFuse.py:620).  g [B,N,C1], p [B,N,1] (after its
    sigmoid), x [B,N,C2], v [B,C2] (after its sigmoid), bp [B,N,C3]."""

    @staticmethod
    def forward(ctx, g, p, x, v, bp):
        B, N, C1 = g.shape
        C2 = x.shape[2] if x is not None else 0
        C3 = bp.shape[2] if bp is not None else 0
        g, p = _contig(g), _contig(p)
        x, v, bp = (_contig(t) if t is not None else None for t in (x, v, bp))
        out = torch.empty((B, N, C1 + C2 + C3), dtype=F32, device=g.device)
        with _dev_ctx(g):
            check(L.lib().mdv_gate_cat_fwd(ptr(g), ptr(p), ptr(x), ptr(v), ptr(bp), ptr(out), B * N, C1, C2, C3, N, L.stream()), "mdv_gate_cat_fwd")
        ctx.save_for_backward(g, p, x, v)
        ctx.meta = (B, N, C1, C2, C3)
        return out

    @staticmethod
    def backward(ctx, dout):
        g, p, x, v = ctx.saved_tensors
        B, N, C1, C2, C3 = ctx.meta
        dev = dout.device
        dout = _contig(dout.float())
        dg = torch.empty((B, N, C1), dtype=F32, device=dev)
        dp = torch.empty((B, N, 1), dtype=F32, device=dev)
        dx = torch.empty((B, N, C2), dtype=F32, device=dev) if C2 else None
        dv = torch.empty((B, C2), dtype=F32, device=dev) if C2 else None
        dbp = torch.empty((B, N, C3), dtype=F32, device=dev) if C3 else None
        with _dev_ctx(dout):
            check(L.lib().mdv_gate_cat_bwd(ptr(dout), ptr(g), ptr(p), ptr(x), ptr(v), ptr(dg), ptr(dp), ptr(dx), ptr(dv), ptr(dbp), B * N, C1, C2, C3,
                                           N, L.stream()), "mdv_gate_cat_bwd")
        return dg, dp, dx, dv, dbp


class ChannelPoolFn(torch.autograd.Function):
    """ChannelPool (TransFuse.py:20-22) on an NHWC map: [B,N,C] -> [B,N,2] = (max over channels, mean over channels)."""

    @staticmethod
    def forward(ctx, x):
        B, N, C = x.shape
        x = _contig(x)
        out = torch.empty((B, N, 2), dtype=F32, device=x.device)
        arg = torch.empty((B, N), dtype=torch.int32, device=x.device)
        with _dev_ctx(x):
            check(L.lib().mdv_channel_pool_fwd(ptr(x), ptr(out), ptr(arg), B * N, C, L.stream()), "mdv_channel_pool_fwd")
        ctx.save_for_backward(arg)
        ctx.meta = (B, N, C)
        return out

    @staticmethod
    def backward(ctx, dout):
        (arg,) = ctx.saved_tensors
        B, N, C = ctx.meta
        dout = _contig(dout.float())
        dx = torch.empty((B, N, C), dtype=F32, device=dout.device)
        with _dev_ctx(dout):
            check(L.lib().mdv_channel_pool_bwd(ptr(dout), ptr(arg), ptr(dx), B * N, C, L.stream()), "mdv_channel_pool_bwd")
        return dx


class Dropout2dFn(torch.autograd.Function):
    """nn.Dropout2d on an NHWC map (TransFuse.py:217,226-245): whole (sample, channel) planes; the mask is regenerated in backward
    from the counter-based RNG (rng_tensor: seed, step) and this call's stream id."""

    @staticmethod
    def forward(ctx, x, p):
        B, N, C = x.shape
        x = _contig(x)
        sid = new_stream_id()
        out = torch.empty_like(x)
        with _dev_ctx(x):
            check(L.lib().mdv_dropout2d(ptr(x), ptr(out), B * N, C, N, ctypes.c_float(p), ptr(rng_tensor(x.device)), sid, L.stream()), "mdv_dropout2d")
        ctx.meta = (B, N, C, float(p), sid)
        return out

    @staticmethod
    def backward(ctx, dout):
        B, N, C, p, sid = ctx.meta
        dout = _contig(dout.float())
        dx = torch.empty_like(dout)
        with _dev_ctx(dout):
            check(L.lib().mdv_dropout2d(ptr(dout), ptr(dx), B * N, C, N, ctypes.c_float(p), ptr(rng_tensor(dout.device)), sid, L.stream()), "mdv_dropout2d")
        return dx, None
