"""MDViT / BASE nn.Modules with the reference's constructor, forward signature, parameter names and state_dict layout
(Models/Transformer/mdvit.py:474-730, Models/Transformer/base.py:340-512), executing on the sm_100a kernels of
libmdvit_b200.so.  The torch.nn layers instantiated here (Conv2d, Linear, LayerNorm, BatchNorm2d) are parameter
CONTAINERS only — their own forward is never called; all arithmetic goes through mdvit_b200.ops.

Drop-in use with the unmodified trainer: put `<repo>/dropin` in front of the reference root on PYTHONPATH so that
`from Models.Transformer.mdvit import MDViT` (multi_train_MDViT.py:58) resolves to this class.  See INTEGRATION.md.
"""
import math
from functools import partial

import torch
from torch import nn

from . import ops

CRPE_WINDOW = {3: 2, 5: 3, 7: 3}


def _ctor_draw(*convs):
    """The reference's conv containers re-draw their conv weights at construction time (mpvit.py:109-113, mdvit.py:104-112,
    Decoders.py:45-53) before MDViT._init_weights overwrites them again.  The values are dead, but the draws advance the
    torch RNG; repeating them keeps `torch.manual_seed(s); MDViT(...)` bit-identical to the reference's random init."""
    for c in convs:
        fan_out = c.kernel_size[0] * c.kernel_size[1] * c.out_channels
        c.weight.data.normal_(0, math.sqrt(2.0 / fan_out))


def _pick(mods, d):
    """The norm of domain d; for the stacked multi-domain pass (d = the G domain keys) the list of the G domains' norms."""
    return [mods[int(k)] for k in d] if isinstance(d, (list, tuple)) else mods[int(d)]


def _norm_args(*norms):
    """The (bufs, trailing norm arguments) of an ops norm Function (see ops._norm_slots).  Each of `norms` is one norm module, or
    the list of the S modules the row groups of a stacked pass use.  Both are set-major, and within a set follow `norms`: the
    (weight, bias) of every norm, and the running buffers of every BatchNorm."""
    sets = list(zip(*(n if isinstance(n, list) else [n] for n in norms)))
    params = tuple(t for s in sets for n in s for t in (n.weight, n.bias))
    bufs = tuple(t for s in sets for n in s if isinstance(n, nn.BatchNorm2d) for t in (n.running_mean, n.running_var, n.num_batches_tracked))
    return bufs, params


# ----------------------------------------------------------------------------------------------- parameter containers
class Conv2d_BN(nn.Module):
    """mpvit.py:81-124 (conv no bias + BN + act)."""

    def __init__(self, in_ch, out_ch, kernel_size=1, stride=1, pad=0, act_layer=None):
        super().__init__()
        self.conv = nn.Conv2d(in_ch, out_ch, kernel_size, stride, pad, bias=False)
        self.bn = nn.BatchNorm2d(out_ch)
        _ctor_draw(self.conv)
        self.act_layer = act_layer() if act_layer is not None else nn.Identity()

    def norm(self, d=None):
        return self.bn


class Conv2d_BN_M(nn.Module):
    """mdvit.py:23-71: Conv2d_BN with one BatchNorm per domain (`bns[int(d)]`)."""

    def __init__(self, in_ch, out_ch, kernel_size=1, stride=1, pad=0, act_layer=None, num_domains=1):
        super().__init__()
        self.conv = nn.Conv2d(in_ch, out_ch, kernel_size, stride, pad, bias=False)
        self.bns = nn.ModuleList([nn.BatchNorm2d(out_ch) for _ in range(num_domains)])
        _ctor_draw(self.conv)
        self.act_layer = act_layer() if act_layer is not None else nn.Identity()

    def norm(self, d=None):
        return _pick(self.bns, d)


class DWConv2d_BN(nn.Module):
    """mdvit.py:74-123: depthwise (groups=in_ch) + pointwise in->out + BN + Hardswish."""

    def __init__(self, in_ch, out_ch, kernel_size=3, stride=1, num_domains=None):
        super().__init__()
        self.dwconv = nn.Conv2d(in_ch, in_ch, kernel_size, stride, (kernel_size - 1) // 2, groups=in_ch, bias=False)
        self.pwconv = nn.Conv2d(in_ch, out_ch, 1, 1, 0, bias=False)
        if num_domains is None:
            self.bn = nn.BatchNorm2d(out_ch)
        else:       # DWConv2d_BN_M, mdvit.py:127-180: domain-specific norms
            self.bns = nn.ModuleList([nn.BatchNorm2d(out_ch) for _ in range(num_domains)])
        self.act = nn.Hardswish()
        self.stride = stride
        _ctor_draw(self.dwconv, self.pwconv)

    def norm(self, d=None):
        return self.bn if hasattr(self, "bn") else _pick(self.bns, d)


class DWCPatchEmbed(nn.Module):
    """mdvit.py:183-208."""

    def __init__(self, in_chans, embed_dim, patch_size=3, stride=1, num_domains=None):
        super().__init__()
        self.patch_conv = DWConv2d_BN(in_chans, embed_dim, patch_size, stride, num_domains)

    def forward(self, x, H, W, after_stem=False, d=None):
        pc = self.patch_conv
        bufs, norm = _norm_args(pc.norm(d))
        y = ops.PatchEmbedFn.apply(x, pc.dwconv.weight, pc.pwconv.weight, bufs, H, W, pc.stride, self.training, after_stem, *norm)
        s = pc.stride
        return y, (H + 2 - 3) // s + 1, (W + 2 - 3) // s + 1


class DecoderDWConv2d_BN(nn.Module):
    """Decoders.py:15-63: 3x3 conv groups=out_ch over 2*out_ch inputs, pointwise out->out, BN, Hardswish."""

    def __init__(self, in_ch, out_ch, num_domains=None):
        super().__init__()
        self.dwconv = nn.Conv2d(in_ch, out_ch, 3, 1, 1, groups=out_ch, bias=False)
        self.pwconv = nn.Conv2d(out_ch, out_ch, 1, 1, 0, bias=False)
        if num_domains is None:
            self.bn = nn.BatchNorm2d(out_ch)
        else:       # Decoders.DWConv2d_BN_M, Decoders.py:66-118
            self.bns = nn.ModuleList([nn.BatchNorm2d(out_ch) for _ in range(num_domains)])
        self.act = nn.Hardswish()
        _ctor_draw(self.dwconv, self.pwconv)

    def norm(self, d=None):
        return self.bn if hasattr(self, "bn") else _pick(self.bns, d)


class ConvPosEnc(nn.Module):
    """mpvit.py:229-248."""

    def __init__(self, dim, k=3):
        super().__init__()
        self.proj = nn.Conv2d(dim, dim, k, 1, k // 2, groups=dim)


class ConvRelPosEnc(nn.Module):
    """mpvit.py:251-318."""

    def __init__(self, Ch, h, window):
        super().__init__()
        self.conv_list = nn.ModuleList()
        self.head_splits = []
        for cur_window, cur_head_split in window.items():
            self.conv_list.append(nn.Conv2d(cur_head_split * Ch, cur_head_split * Ch, cur_window, padding=cur_window // 2,
                                            groups=cur_head_split * Ch))
            self.head_splits.append(cur_head_split)


class FactorAtt_ConvRelPosEnc(nn.Module):
    """mpvit.py:321-373 (no domain adapter)."""

    def __init__(self, dim, num_heads=8, qkv_bias=False, attn_drop=0.0, proj_drop=0.0, shared_crpe=None):
        super().__init__()
        self.num_heads = num_heads
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.attn_drop = nn.Dropout(attn_drop)  # constructed but never applied by the reference either
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)
        self.crpe = shared_crpe
        self.domain_layer = None


class FactorAtt_ConvRelPosEnc_Sup(nn.Module):
    """mdvit.py:243-313 (DA: domain_layer MLP -> softmax over heads gate)."""

    def __init__(self, dim, num_heads=8, qkv_bias=False, attn_drop=0.0, proj_drop=0.0, shared_crpe=None, r=2, num_domains=4):
        super().__init__()
        self.num_heads = num_heads
        hidden_dim = max(dim // r, 4)
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)
        self.domain_layer = nn.Sequential(nn.Linear(num_domains, hidden_dim), nn.ReLU(inplace=True), nn.Linear(hidden_dim, dim))
        self.crpe = shared_crpe


class Mlp(nn.Module):
    """mpvit.py:51-78."""

    def __init__(self, in_features, hidden_features, drop=0.0):
        super().__init__()
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.act = nn.GELU()
        self.fc2 = nn.Linear(hidden_features, in_features)
        self.drop = nn.Dropout(drop)


class SerialBlock_adapt(nn.Module):
    """mdvit.py:316-361."""

    def __init__(self, dim, num_heads, mlp_ratio, qkv_bias, drop, attn_drop, drop_path, norm_layer, shared_cpe, shared_crpe,
                 adapt_method, num_domains, label_only_guard=False, dsn=False):
        super().__init__()
        self.label_only_guard = label_only_guard   # base.py:216 tests only `domain_label != None`
        if num_heads != ops.HEADS:
            raise ValueError("mdvit_b200 kernels are specialised for 8 attention heads (the reference's only setting)")
        self.cpe = shared_cpe
        self.dsn = dsn          # SerialBlock_adapt_M (mdvit.py:364-412): norm1s / norm2s, one LayerNorm per domain
        if dsn:
            self.norm1s = nn.ModuleList([norm_layer(dim) for _ in range(num_domains)])
        else:
            self.norm1 = norm_layer(dim)
        self.adapt_method = adapt_method
        if adapt_method == 'Sup':
            self.factoratt_crpe = FactorAtt_ConvRelPosEnc_Sup(dim, num_heads, qkv_bias, attn_drop, drop, shared_crpe,
                                                              num_domains=num_domains)
        else:
            self.factoratt_crpe = FactorAtt_ConvRelPosEnc(dim, num_heads, qkv_bias, attn_drop, drop, shared_crpe)
        self.drop_path = nn.Identity()
        self.drop_path_rate = float(drop_path)
        self.drop_rate = float(drop)
        if dsn:
            self.norm2s = nn.ModuleList([norm_layer(dim) for _ in range(num_domains)])
        else:
            self.norm2 = norm_layer(dim)
        self.mlp = Mlp(dim, int(dim * mlp_ratio), drop)

    def forward(self, x, size, domain_label=None, d=None):
        H, W = size
        norm1 = _pick(self.norm1s, d) if self.dsn else self.norm1
        norm2 = _pick(self.norm2s, d) if self.dsn else self.norm2
        _, norm = _norm_args(norm1, norm2)
        att = self.factoratt_crpe
        # dispatch quirks of mdvit.py:350-353 preserved: Sup attention needs a label, plain attention rejects one
        use_label = domain_label is not None and (self.label_only_guard or self.adapt_method is not None)
        if att.domain_layer is not None and not use_label:
            raise TypeError("FactorAtt_ConvRelPosEnc_Sup.forward() missing 1 required positional argument: 'domain_label'")
        if att.domain_layer is None and use_label:
            raise TypeError("FactorAtt_ConvRelPosEnc.forward() takes 3 positional arguments but 4 were given")
        dl = att.domain_layer
        da = (dl[0].weight, dl[0].bias, dl[2].weight, dl[2].bias) if dl is not None else (None, None, None, None)
        cl = att.crpe.conv_list
        n1 = self.norm1s[0] if self.dsn else self.norm1
        if not (isinstance(n1, nn.LayerNorm) and abs(n1.eps - 1e-6) < 1e-12):
            raise ValueError("mdvit_b200 supports norm_layer=LayerNorm(eps=1e-6) (the reference default)")
        return ops.BlockFn.apply(
            x, domain_label if use_label else None, self.cpe.proj.weight, self.cpe.proj.bias,
            cl[0].weight, cl[0].bias, cl[1].weight, cl[1].bias, cl[2].weight, cl[2].bias,
            att.qkv.weight, att.qkv.bias, att.proj.weight, att.proj.bias, da[0], da[1], da[2], da[3],
            self.mlp.fc1.weight, self.mlp.fc1.bias, self.mlp.fc2.weight, self.mlp.fc2.bias,
            H, W, self.drop_rate, self.drop_path_rate, self.training, *norm)


class MHSA_stage_adapt(nn.Module):
    """mdvit.py:415-440: one shared ConvPosEnc + ConvRelPosEnc, `num_layers` serial blocks."""

    def __init__(self, dim, num_layers, num_heads, mlp_ratio, qkv_bias=True, drop_rate=0., attn_drop_rate=0., drop_path_rate=0.,
                 num_domains=4, norm_layer=nn.LayerNorm, adapt_method=None, label_only_guard=False, dsn=False):
        super().__init__()
        self.cpe = ConvPosEnc(dim, k=3)
        self.crpe = ConvRelPosEnc(Ch=dim // num_heads, h=num_heads, window=CRPE_WINDOW)
        self.mhca_blks = nn.ModuleList([
            SerialBlock_adapt(dim, num_heads, mlp_ratio, qkv_bias, drop_rate, attn_drop_rate, drop_path_rate, norm_layer,
                              self.cpe, self.crpe, adapt_method, num_domains, label_only_guard, dsn) for _ in range(num_layers)])

    def forward(self, x, H, W, domain_label=None, d=None):
        for blk in self.mhca_blks:
            x = blk(x, (H, W), domain_label, d)
        return x


class UnetDecodingBlockTransformer(nn.Module):
    """Decoders.py:174-214 (use_res=False)."""

    def __init__(self, in_channel, out_channel, mhsa_block, num_domains=None):
        super().__init__()
        self.conv_before = nn.Conv2d(in_channel, out_channel, kernel_size=1)
        self.conv_after = DecoderDWConv2d_BN(out_channel * 2, out_channel, num_domains)
        self.mhsa_block = mhsa_block

    def forward(self, x, h, w, skip, H, W, domain_label=None, d=None):
        ca = self.conv_after
        bufs, norm = _norm_args(ca.norm(d))
        out = ops.DecoderConvFn.apply(x, skip, self.conv_before.weight, self.conv_before.bias, ca.dwconv.weight, ca.pwconv.weight,
                                      bufs, h, w, H, W, self.training, *norm)
        return self.mhsa_block(out, H, W, domain_label, d)


class MLPDecoderFM(nn.Module):
    """Decoders.py:289-339."""

    with_feature = True      # MLPDecoderFM also consumes the main decoder's last feature map (x5)

    def __init__(self, in_channels, out_channel, hidden_channel=256, outfeature_channel=64, dropout_ratio=0.1):
        super().__init__()
        if out_channel != 1:
            raise ValueError("mdvit_b200 implements the single-class head used by the reference trainers")
        if not self.with_feature:
            outfeature_channel = 0
        self.linear1 = nn.Conv2d(in_channels[0], hidden_channel, 1)
        self.linear2 = nn.Conv2d(in_channels[1], hidden_channel, 1)
        self.linear3 = nn.Conv2d(in_channels[2], hidden_channel, 1)
        self.linear4 = nn.Conv2d(in_channels[3], hidden_channel, 1)
        self.linear_fuse = nn.Sequential(nn.Conv2d(hidden_channel * 4 + outfeature_channel, hidden_channel, 1),
                                         nn.BatchNorm2d(hidden_channel), nn.ReLU(inplace=True))
        self.dropout = nn.Dropout2d(dropout_ratio)
        self.linear_out = nn.Conv2d(hidden_channel, out_channel, 1)
        self.avg_pool = nn.AdaptiveAvgPool2d((1, 1))

    def forward(self, feats, sizes, img_size):
        x1, x2, x3, x4 = feats[:4]
        x5 = feats[4] if self.with_feature else None
        bn = self.linear_fuse[1]
        return ops.AuxFn.apply(x1, x2, x3, x4, x5, self.linear1.weight, self.linear1.bias, self.linear2.weight, self.linear2.bias,
                               self.linear3.weight, self.linear3.bias, self.linear4.weight, self.linear4.bias,
                               self.linear_fuse[0].weight, self.linear_fuse[0].bias, bn.weight, bn.bias, self.linear_out.weight,
                               self.linear_out.bias, (bn.running_mean, bn.running_var, bn.num_batches_tracked), tuple(sizes),
                               int(img_size[0]), int(img_size[1]), float(self.dropout.p), self.training)


class MLPDecoder(MLPDecoderFM):
    """Decoders.py:239-286: the SegFormer-style auxiliary decoder WITHOUT the main-decoder feature (decoder_name='MLP')."""
    with_feature = False

    def __init__(self, in_channels, out_channel, hidden_channel=256, dropout_ratio=0.1):
        super().__init__(in_channels, out_channel, hidden_channel, 0, dropout_ratio)


class ASPPConv(nn.Sequential):
    """Utils/_deeplab.py:115-122."""

    def __init__(self, in_channels, out_channels, dilation):
        super().__init__(nn.Conv2d(in_channels, out_channels, 3, padding=dilation, dilation=dilation, bias=False),
                         nn.BatchNorm2d(out_channels), nn.ReLU(inplace=True))


class ASPPPooling(nn.Sequential):
    """Utils/_deeplab.py:124-135."""

    def __init__(self, in_channels, out_channels):
        super().__init__(nn.AdaptiveAvgPool2d(1), nn.Conv2d(in_channels, out_channels, 1, bias=False), nn.BatchNorm2d(out_channels),
                         nn.ReLU(inplace=True))


class ASPP(nn.Module):
    """Utils/_deeplab.py:137-165 (parameter container; the arithmetic is ops.DeepLabFn)."""

    def __init__(self, in_channels, atrous_rates):
        super().__init__()
        out_channels = 256
        modules = [nn.Sequential(nn.Conv2d(in_channels, out_channels, 1, bias=False), nn.BatchNorm2d(out_channels), nn.ReLU(inplace=True))]
        modules += [ASPPConv(in_channels, out_channels, r) for r in tuple(atrous_rates)]
        modules.append(ASPPPooling(in_channels, out_channels))
        self.convs = nn.ModuleList(modules)
        self.project = nn.Sequential(nn.Conv2d(5 * out_channels, out_channels, 1, bias=False), nn.BatchNorm2d(out_channels),
                                     nn.ReLU(inplace=True), nn.Dropout(0.1))
        self.atrous_rates = tuple(atrous_rates)


class DeepLabV3Decoder(nn.Module):
    """Decoders.py:218-235: ASPP(512, [6,12,18]) -> 3x3 conv -> BN -> ReLU -> 1x1 conv on the LAST encoder map, resized to the
    image.  Called like the other auxiliary decoders (token-major feature list + their sizes)."""

    with_feature = False

    def __init__(self, in_channel, out_channel, aspp_dilate=[6, 12, 18], conv_norm=nn.BatchNorm2d):
        super().__init__()
        if conv_norm is not nn.BatchNorm2d or out_channel != 1:
            raise ValueError("mdvit_b200 implements DeepLabV3Decoder(in_channel, 1) with BatchNorm2d")
        self.classifier = nn.Sequential(ASPP(in_channel, aspp_dilate), nn.Conv2d(256, 256, 3, padding=1, bias=False), conv_norm(256),
                                        nn.ReLU(inplace=True), nn.Conv2d(256, out_channel, 1))

    def forward(self, feats, sizes, img_size):
        x, (H, W) = feats[3], sizes[3]          # `feature[-1]` of the four encoder maps (mdvit.py:715-722, Decoders.py:230-231)
        aspp, conv, bn, _, fc = self.classifier
        pairs = [(aspp.convs[0][0], aspp.convs[0][1]), (aspp.convs[1][0], aspp.convs[1][1]), (aspp.convs[2][0], aspp.convs[2][1]),
                 (aspp.convs[3][0], aspp.convs[3][1]), (aspp.convs[4][1], aspp.convs[4][2]), (aspp.project[0], aspp.project[1]), (conv, bn)]
        wgb, bufs = [], []
        for c, n in pairs:
            wgb += [c.weight, n.weight, n.bias]
            bufs.append((n.running_mean, n.running_var, n.num_batches_tracked))
        y = ops.DeepLabFn.apply(x, H, W, aspp.atrous_rates, float(aspp.project[3].p), self.training, bufs, *wgb)
        return ops.HeadFn.apply(y, fc.weight, fc.bias, H, W, int(img_size[0]), int(img_size[1]))


AUX_DECODERS = {'MLPFM': MLPDecoderFM, 'MLP': MLPDecoder}


# ----------------------------------------------------------------------------------------------- models
class _Trunk(nn.Module):
    """Shared encoder / bridge / decoder of MDViT and BASE."""

    def _build_trunk(self, in_chans, num_stages, num_layers, embed_dims, mlp_ratios, num_heads, qkv_bias, drop_rate, attn_drop_rate,
                     drop_path_rate, norm_layer, conv_norm, adapt_method, num_domains, label_only_guard=False):
        if num_stages != 4 or in_chans != 3:
            raise ValueError("mdvit_b200 implements the 4-stage, 3-channel configuration of the reference trainers")
        if conv_norm is not nn.BatchNorm2d:
            raise ValueError("mdvit_b200 implements conv_norm=nn.BatchNorm2d (the reference trainers' setting)")
        self.num_stages = num_stages
        self.embed_dims = list(embed_dims)
        self.stem = nn.Sequential(
            Conv2d_BN(in_chans, embed_dims[0] // 2, 3, 2, 1, act_layer=nn.Hardswish),
            Conv2d_BN(embed_dims[0] // 2, embed_dims[0], 3, 2, 1, act_layer=nn.Hardswish))
        self.patch_embed_stages = nn.ModuleList([
            DWCPatchEmbed(embed_dims[idx] if idx == 0 else embed_dims[idx - 1], embed_dims[idx], 3, 1 if idx == 0 else 2)
            for idx in range(num_stages)])

        def stage(idx):
            return MHSA_stage_adapt(embed_dims[idx], num_layers[idx], num_heads[idx], mlp_ratios[idx], qkv_bias, drop_rate,
                                    attn_drop_rate, drop_path_rate, num_domains, norm_layer, adapt_method, label_only_guard)

        self.mhsa_stages = nn.ModuleList([stage(idx) for idx in range(num_stages)])
        self.bridge = nn.Sequential(
            nn.Conv2d(embed_dims[3], embed_dims[3], 3, 1, 1), nn.BatchNorm2d(embed_dims[3]), nn.ReLU(inplace=True),
            nn.Conv2d(embed_dims[3], embed_dims[3] * 2, 3, 1, 1), nn.BatchNorm2d(embed_dims[3] * 2), nn.ReLU(inplace=True))
        self.mhsa_list = [stage(idx) for idx in range(num_stages)]   # plain list, as in mdvit.py:568
        self.decoder1 = UnetDecodingBlockTransformer(embed_dims[3] * 2, embed_dims[3], self.mhsa_list[3])
        self.decoder2 = UnetDecodingBlockTransformer(embed_dims[3], embed_dims[2], self.mhsa_list[2])
        self.decoder3 = UnetDecodingBlockTransformer(embed_dims[2], embed_dims[1], self.mhsa_list[1])
        self.decoder4 = UnetDecodingBlockTransformer(embed_dims[1], embed_dims[0], self.mhsa_list[0])
        self.finalconv = nn.Sequential(nn.Conv2d(embed_dims[0], 1, kernel_size=1))

    def _init_weights(self, m):
        """mdvit.py:648-664."""
        if isinstance(m, nn.Linear):
            nn.init.trunc_normal_(m.weight, std=.02)
            if m.bias is not None:
                nn.init.constant_(m.bias, 0)
        elif isinstance(m, nn.LayerNorm):
            nn.init.constant_(m.bias, 0)
            nn.init.constant_(m.weight, 1.0)
        elif isinstance(m, nn.Conv2d):
            fan_out = m.kernel_size[0] * m.kernel_size[1] * m.out_channels
            fan_out //= m.groups
            m.weight.data.normal_(0, math.sqrt(2.0 / fan_out))
            if m.bias is not None:
                m.bias.data.zero_()
        elif isinstance(m, nn.BatchNorm2d):
            m.weight.data.fill_(1)
            m.bias.data.zero_()

    def _stem_parts(self, d=None):
        return self.stem[0].conv, self.stem[0].bn, self.stem[1].conv, self.stem[1].bn

    def _bridge_parts(self, d=None):
        b = self.bridge
        return b[0], b[1], b[3], b[4]

    def _trunk_forward(self, x, domain_label, d=None):
        if x.dim() != 4 or x.shape[1] != 3 or x.shape[2] % 32 or x.shape[3] % 32:
            raise ValueError("input must be [B,3,H,W] with H and W divisible by 32")
        if not x.is_cuda:
            raise RuntimeError("mdvit_b200 runs on CUDA (sm_100a) only; there is no CPU path")
        c0, n0, c1, n1 = self._stem_parts(d)
        H, W = x.shape[2] // 4, x.shape[3] // 4
        bufs, norm = _norm_args(n0, n1)
        t = ops.StemFn.apply(x, c0.weight, c1.weight, bufs, self.training, *norm)
        enc = []
        for idx in range(self.num_stages):
            t, H, W = self.patch_embed_stages[idx](t, H, W, after_stem=(idx == 0), d=d)
            t = self.mhsa_stages[idx](t, H, W, domain_label, d)
            enc.append((t, H, W))
        return enc

    def _bridge(self, enc, d=None):
        t3, H3, W3 = enc[3]
        c0, n0, c1, n1 = self._bridge_parts(d)
        bufs, norm = _norm_args(n0, n1)
        return ops.BridgeFn.apply(t3, c0.weight, c0.bias, c1.weight, c1.bias, bufs, H3, W3, self.training, *norm)

    def _decode_from(self, out, enc, decoders, domain_label, d=None):
        h, w = enc[3][1], enc[3][2]
        for dec, (skip, H, W) in zip(decoders, (enc[3], enc[2], enc[1], enc[0])):
            out = dec(out, h, w, skip, H, W, domain_label, d)
            h, w = H, W
        return out, h, w

    def _decode(self, enc, domain_label, d=None):
        return self._decode_from(self._bridge(enc, d), enc, (self.decoder1, self.decoder2, self.decoder3, self.decoder4), domain_label, d)

    def _head(self, dec4, h, w, img_size):
        fc = self.finalconv[0]
        return ops.HeadFn.apply(dec4, fc.weight, fc.bias, h, w, int(img_size[0]), int(img_size[1]))


class MDViT(_Trunk):
    """Drop-in for Models.Transformer.mdvit.MDViT (decoder_name='MLPFM')."""

    def __init__(self, img_size=512, in_chans=3, num_stages=4, num_layers=[2, 2, 2, 2], embed_dims=[64, 128, 320, 512],
                 mlp_ratios=[8, 8, 4, 4], num_heads=[8, 8, 8, 8], qkv_bias=True, qk_scale=None, drop_rate=0., attn_drop_rate=0.,
                 drop_path_rate=0.0, norm_layer=partial(nn.LayerNorm, eps=1e-6), conv_norm=nn.BatchNorm2d, adapt_method=None,
                 num_domains=4, decoder_name='MLPFM', **kwargs):
        super().__init__()
        if qk_scale is not None:
            raise ValueError("mdvit_b200 implements qk_scale=None (head_dim**-0.5), the reference trainers' setting")
        if decoder_name not in AUX_DECODERS and decoder_name not in ('Transformer', 'DeepLabV3'):
            raise NotImplementedError("mdvit_b200 implements decoder_name in ('MLPFM', 'MLP', 'DeepLabV3', 'Transformer') (mdvit.py:594-642)")
        self.decoder_name = decoder_name
        self._build_trunk(in_chans, num_stages, num_layers, embed_dims, mlp_ratios, num_heads, qkv_bias, drop_rate, attn_drop_rate,
                          drop_path_rate, norm_layer, conv_norm, adapt_method, num_domains)
        if decoder_name == 'Transformer':
            # mdvit.py:613-642: one more transformer decoder (4 stages without the domain adapter + a 1x1 head) per domain
            debranchs = []
            for _ in range(num_domains):
                mh = [MHSA_stage_adapt(embed_dims[idx], num_layers[idx], num_heads[idx], mlp_ratios[idx], qkv_bias, drop_rate,
                                       attn_drop_rate, drop_path_rate, num_domains, norm_layer, False) for idx in range(num_stages)]
                debranchs.append(nn.ModuleList([
                    UnetDecodingBlockTransformer(embed_dims[3] * 2, embed_dims[3], mh[3]),
                    UnetDecodingBlockTransformer(embed_dims[3], embed_dims[2], mh[2]),
                    UnetDecodingBlockTransformer(embed_dims[2], embed_dims[1], mh[1]),
                    UnetDecodingBlockTransformer(embed_dims[1], embed_dims[0], mh[0]),
                    nn.Sequential(nn.Conv2d(embed_dims[0], 1, kernel_size=1))]))
            self.debranchs = nn.ModuleList(debranchs)
        elif decoder_name == 'DeepLabV3':
            self.debranch1 = DeepLabV3Decoder(512, 1)
            self.debranch2 = DeepLabV3Decoder(512, 1)
            self.debranch3 = DeepLabV3Decoder(512, 1)
            self.debranch4 = DeepLabV3Decoder(512, 1)
        else:
            Aux = AUX_DECODERS[decoder_name]
            self.debranch1 = Aux(embed_dims, 1, 512)
            self.debranch2 = Aux(embed_dims, 1, 512)
            self.debranch3 = Aux(embed_dims, 1, 512)
            self.debranch4 = Aux(embed_dims, 1, 512)
        # Inference-only switch (not a constructor argument: the signature stays the reference's).  The reference's test loop
        # passes `d`, computes the auxiliary decoder (45% of the forward FLOPs) and then uses only output[0]
        # (multi_train_MDViT.py:377-378).  With this flag set, an eval-mode forward returns [out, None] even when `d` is given.
        self.skip_aux_in_eval = False
        self.apply(self._init_weights)

    def forward(self, x, domain_label=None, d=None, out_feat=False, out_seg=True):
        img_size = x.shape[2:]
        enc = self._trunk_forward(x, domain_label)
        if not out_seg:
            return {'seg': None, 'feat': enc[3][0].mean(dim=1)}
        bridge_out = self._bridge(enc)
        dec4, h, w = self._decode_from(bridge_out, enc, (self.decoder1, self.decoder2, self.decoder3, self.decoder4), domain_label)
        out = self._head(dec4, h, w, img_size)
        aux_out = None
        if self.decoder_name == 'Transformer':
            branch = self.debranchs[int(d)]          # (mdvit.py:704-706: int(d) is unconditional for this decoder)
            if self.training or not self.skip_aux_in_eval:
                aux_out = self._transformer_aux(branch, bridge_out, enc, img_size)
        elif d in ('0', '1', '2', '3') and (self.training or not self.skip_aux_in_eval):
            branch = getattr(self, f'debranch{int(d) + 1}')
            feats = [e[0] for e in enc] + [dec4]
            aux_out = branch(feats, [(e[1], e[2]) for e in enc], img_size)
        if out_feat:
            return {'seg': [out, aux_out], 'feat': enc[3][0].mean(dim=1)}
        return [out, aux_out]

    def _transformer_aux(self, branch, bridge_out, enc, img_size):
        """mdvit.py:704-712: the per-domain transformer decoder on the shared bridge output and encoder skips (no DA gate)."""
        a4, h, w = self._decode_from(bridge_out, enc, (branch[0], branch[1], branch[2], branch[3]), None)
        fc = branch[4][0]
        return ops.HeadFn.apply(a4, fc.weight, fc.bias, h, w, int(img_size[0]), int(img_size[1]))

    def forward_multi(self, x, domain_label, domains):
        """The G single-domain forwards of one training step (multi_train_MDViT.py:129-146 calls forward once per domain)
        as ONE pass over the stacked batch: x = cat of G equal mini-batches [G*B,3,H,W], domain_label [G*B, num_domains],
        domains = the G domain keys ('0'..'3') in stacking order.  Every trunk kernel runs once on G*B samples (the trunk is
        per-sample except BatchNorm, which is evaluated per group of B samples — ops.bn_groups — exactly as G separate
        forwards would); each domain's auxiliary decoder then runs on its slice.  Returns [(out_d, aux_d)] per domain.
        Equivalent to [self(x_d, label_d, d) for d in domains] up to dropout masks."""
        G = len(domains)
        if x.shape[0] % G:
            raise ValueError("forward_multi needs G equal mini-batches stacked along dim 0")
        B = x.shape[0] // G
        img_size = x.shape[2:]
        with ops.bn_groups(G if self.training else 1):
            enc = self._trunk_forward(x, domain_label)
            bridge_out = self._bridge(enc)
            dec4, h, w = self._decode_from(bridge_out, enc, (self.decoder1, self.decoder2, self.decoder3, self.decoder4), domain_label)
        out = self._head(dec4, h, w, img_size)
        # per-domain slices of the five feature maps the auxiliary decoders read, and of the main logits
        fifth = bridge_out if self.decoder_name == 'Transformer' else dec4
        split = [ops.SplitDomainsFn.apply(t, G) for t in [e[0] for e in enc] + [fifth, out]]
        res = []
        for g, d in enumerate(domains):
            aux_out = None
            if self.decoder_name == 'Transformer':
                enc_g = [(split[i][g], enc[i][1], enc[i][2]) for i in range(4)]
                aux_out = self._transformer_aux(self.debranchs[int(d)], split[4][g], enc_g, img_size)
            elif d in ('0', '1', '2', '3'):
                branch = getattr(self, f'debranch{int(d) + 1}')
                aux_out = branch([split[i][g] for i in range(5)], [(e[1], e[2]) for e in enc], img_size)
            res.append((split[5][g], aux_out))
        return res


class MDViT_DSN(_Trunk):
    """Drop-in for Models.Transformer.mdvit.MDViT_DSN (mdvit.py:735-960): MDViT with DOMAIN-SPECIFIC NORMS — every
    BatchNorm (stem, patch embeddings, bridge, decoder convs) and every LayerNorm (norm1s / norm2s of each block) exists
    once per domain and forward(x, domain_label, d) uses the set `int(d)`.  The kernels are the same: the autograd
    Functions take the norm parameters as arguments, so domain selection is a pointer choice on the host.  In the stacked
    training pass (forward_multi) the choice moves to the device: the norm kernels take one parameter set per row group.
    decoder_name='MLPFM' is the implemented auxiliary decoder (the reference class defaults to 'MLP')."""

    domain_specific_norms = True      # forward needs the domain key d even without auxiliary branches (MKDTrainer passes it)

    def __init__(self, img_size=512, in_chans=3, num_stages=4, num_layers=[2, 2, 2, 2], embed_dims=[64, 128, 320, 512],
                 mlp_ratios=[8, 8, 4, 4], num_heads=[8, 8, 8, 8], qkv_bias=True, qk_scale=None, drop_rate=0., attn_drop_rate=0.,
                 drop_path_rate=0.0, norm_layer=partial(nn.LayerNorm, eps=1e-6), conv_norm=nn.BatchNorm2d, adapt_method=None,
                 num_domains=4, decoder_name='MLP', **kwargs):
        super().__init__()
        if qk_scale is not None or num_stages != 4 or in_chans != 3 or conv_norm is not nn.BatchNorm2d:
            raise ValueError("mdvit_b200 implements the 4-stage, 3-channel, BatchNorm2d configuration of the reference trainers")
        if decoder_name is not None and decoder_name not in AUX_DECODERS:      # (None: BASE_DSN, no auxiliary branches)
            raise NotImplementedError("mdvit_b200 implements decoder_name in ('MLPFM', 'MLP') for MDViT_DSN")
        self.num_stages, self.decoder_name, self.embed_dims = num_stages, decoder_name, list(embed_dims)
        self.stem_1 = Conv2d_BN_M(in_chans, embed_dims[0] // 2, 3, 2, 1, act_layer=nn.Hardswish, num_domains=num_domains)
        self.stem_2 = Conv2d_BN_M(embed_dims[0] // 2, embed_dims[0], 3, 2, 1, act_layer=nn.Hardswish, num_domains=num_domains)
        self.patch_embed_stages = nn.ModuleList([
            DWCPatchEmbed(embed_dims[idx] if idx == 0 else embed_dims[idx - 1], embed_dims[idx], 3, 1 if idx == 0 else 2, num_domains)
            for idx in range(num_stages)])

        def stage(idx):
            return MHSA_stage_adapt(embed_dims[idx], num_layers[idx], num_heads[idx], mlp_ratios[idx], qkv_bias, drop_rate,
                                    attn_drop_rate, drop_path_rate, num_domains, norm_layer, adapt_method, dsn=True)

        self.mhsa_stages = nn.ModuleList([stage(idx) for idx in range(num_stages)])
        self.bridge_conv1 = nn.Conv2d(embed_dims[3], embed_dims[3], 3, 1, 1)
        self.bridge_norms1 = nn.ModuleList([nn.BatchNorm2d(embed_dims[3]) for _ in range(num_domains)])
        self.bridge_act1 = nn.ReLU(inplace=True)
        self.bridge_conv2 = nn.Conv2d(embed_dims[3], embed_dims[3] * 2, 3, 1, 1)
        self.bridge_norms2 = nn.ModuleList([nn.BatchNorm2d(embed_dims[3] * 2) for _ in range(num_domains)])
        self.bridge_act2 = nn.ReLU(inplace=True)
        self.mhsa_list = [stage(idx) for idx in range(num_stages)]
        self.decoder1 = UnetDecodingBlockTransformer(embed_dims[3] * 2, embed_dims[3], self.mhsa_list[3], num_domains)
        self.decoder2 = UnetDecodingBlockTransformer(embed_dims[3], embed_dims[2], self.mhsa_list[2], num_domains)
        self.decoder3 = UnetDecodingBlockTransformer(embed_dims[2], embed_dims[1], self.mhsa_list[1], num_domains)
        self.decoder4 = UnetDecodingBlockTransformer(embed_dims[1], embed_dims[0], self.mhsa_list[0], num_domains)
        self.finalconv = nn.Sequential(nn.Conv2d(embed_dims[0], 1, kernel_size=1))
        if decoder_name is not None:
            Aux = AUX_DECODERS[decoder_name]
            self.debranch1 = Aux(embed_dims, 1, 512)
            self.debranch2 = Aux(embed_dims, 1, 512)
            self.debranch3 = Aux(embed_dims, 1, 512)
            self.debranch4 = Aux(embed_dims, 1, 512)
        self.skip_aux_in_eval = False
        self.apply(self._init_weights)

    def _stem_parts(self, d=None):
        return self.stem_1.conv, self.stem_1.norm(d), self.stem_2.conv, self.stem_2.norm(d)

    def forward_multi(self, x, domain_label, domains):
        """The G single-domain forwards of one training step as ONE pass over the stacked batch (see MDViT.forward_multi):
        x = cat of G equal mini-batches, domain_label the matching rows (or None), domains the G distinct domain keys in stacking
        order.  Row group g is normalised with norm set int(domains[g]) in every BatchNorm (stem, patch embeddings, bridge,
        decoder convs) and LayerNorm (norm1s / norm2s): one kernel launch serves all groups, each group's statistics and
        running buffers are its own, and each set's gradients come from its group only.  The auxiliary decoders run per slice.
        Returns [(out_d, aux_d)] per domain (aux_d None for BASE_DSN); equivalent to the G separate forwards up to dropout masks.
        In eval mode it returns the G separate forwards: folding one BatchNorm set per row group into the GEMM epilogues (the
        single-domain eval path) is not implemented."""
        G = len(domains)
        domains = [str(d) for d in domains]
        if len(set(domains)) != G:
            raise ValueError(f"forward_multi needs distinct domains (each group updates its own norm set), got {domains}")
        if x.shape[0] % G:
            raise ValueError("forward_multi needs G equal mini-batches stacked along dim 0")
        B = x.shape[0] // G
        if not self.training:
            res = []
            for g, d in enumerate(domains):
                o = self(x[g * B:(g + 1) * B], None if domain_label is None else domain_label[g * B:(g + 1) * B], d)
                res.append(tuple(o) if isinstance(o, list) else (o, None))
            return res
        img_size = x.shape[2:]
        with ops.bn_groups(G):
            enc = self._trunk_forward(x, domain_label, domains)
            dec4, h, w = self._decode(enc, domain_label, domains)
        out = self._head(dec4, h, w, img_size)
        if self.decoder_name is None:
            return [(o, None) for o in ops.SplitDomainsFn.apply(out, G)]
        split = [ops.SplitDomainsFn.apply(t, G) for t in [e[0] for e in enc] + [dec4, out]]
        res = []
        for g, d in enumerate(domains):
            aux_out = None
            if d in ('0', '1', '2', '3'):
                branch = getattr(self, f'debranch{int(d) + 1}')
                aux_out = branch([split[i][g] for i in range(5)], [(e[1], e[2]) for e in enc], img_size)
            res.append((split[5][g], aux_out))
        return res

    def _bridge_parts(self, d=None):
        return self.bridge_conv1, _pick(self.bridge_norms1, d), self.bridge_conv2, _pick(self.bridge_norms2, d)

    def _sample_sets(self, domains, B, device):
        """domains -> the int32 [B] CUDA vector of per-sample norm sets.  Sequences and CPU tensors are checked here (length, range,
        integer keys); a CUDA tensor is only checked for length and dtype and converted on the device, never read back, so the call
        stays graph-capturable (an out-of-range value there gives NaN rows, see mdv_gemm_nt_tf32_sets)."""
        S = len(self.stem_1.bns)
        if torch.is_tensor(domains):
            if domains.dim() != 1 or domains.shape[0] != B:
                raise ValueError(f"forward_mixed needs one domain per sample: {B} samples, domains of shape {tuple(domains.shape)}")
            if domains.dtype.is_floating_point or domains.dtype.is_complex or domains.dtype == torch.bool:
                raise TypeError(f"forward_mixed needs integer domain keys, got {domains.dtype}")
            if domains.is_cuda:
                return domains.to(device=device, dtype=torch.int32).contiguous()
            keys = [int(k) for k in domains.tolist()]
        else:
            domains = list(domains)
            if len(domains) != B:
                raise ValueError(f"forward_mixed needs one domain per sample: {B} samples, {len(domains)} domains")
            keys = []
            for k in domains:
                if isinstance(k, bool) or not isinstance(k, (int, str)) or (isinstance(k, str) and not k.strip().lstrip("-").isdigit()):
                    raise TypeError(f"forward_mixed domain keys are ints or integer strings, got {k!r}")
                keys.append(int(k))
        bad = [k for k in keys if not 0 <= k < S]
        if bad:
            raise ValueError(f"domain keys must lie in [0, {S}): got {bad}")
        return torch.tensor(keys, dtype=torch.int32).to(device)

    def forward_mixed(self, x, domain_label, domains):
        """Inference on a batch that mixes domains: sample b is normalised with norm set int(domains[b]) in every BatchNorm and
        LayerNorm, in ONE trunk, bridge, decoder and head pass (the norm kernels read the set index per sample on the device; see
        ops.norm_sets).  Equivalent to forward(x[b:b+1], domain_label[b:b+1], str(domains[b]))[0] per sample.
        domains: one key per sample — a sequence of str / int, a CPU integer tensor, or a CUDA integer tensor of length B (the
        last is never read back: write new keys into a captured tensor and replay the graph).  domain_label follows forward's
        rule (required for adapt_method='Sup', None otherwise).  Returns the main logits [B, 1, H, W]; the auxiliary decoders do
        not run (the reference's test loop discards them, multi_train_MDViT.py:377-378).  Eval mode only."""
        if self.training:
            raise RuntimeError("forward_mixed is an inference path (eval mode); the multi-domain training pass is forward_multi")
        S = len(self.stem_1.bns)
        if S > 8:
            raise ValueError(f"forward_mixed supports up to 8 norm sets (MDV_MAX_GROUPS), the model has {S}")
        if x.dim() != 4:
            raise ValueError("input must be [B,3,H,W]")
        sample_set = self._sample_sets(domains, x.shape[0], x.device)
        if not x.is_cuda:
            raise RuntimeError("mdvit_b200 runs on CUDA (sm_100a) only; there is no CPU path")
        keys = [str(i) for i in range(S)]
        img_size = x.shape[2:]
        with ops.norm_sets(sample_set):
            enc = self._trunk_forward(x, domain_label, keys)
            dec4, h, w = self._decode(enc, domain_label, keys)
            return self._head(dec4, h, w, img_size)

    def forward(self, x, domain_label=None, d=None, out_feat=False, out_seg=True):
        img_size = x.shape[2:]
        int(d)      # the reference indexes its norm lists with int(d) everywhere (mdvit.py:65,398,917): d is required
        enc = self._trunk_forward(x, domain_label, d)
        if not out_seg:
            return {'seg': None, 'feat': enc[3][0].mean(dim=1)}
        dec4, h, w = self._decode(enc, domain_label, d)
        out = self._head(dec4, h, w, img_size)
        aux_out = None
        if d in ('0', '1', '2', '3') and (self.training or not self.skip_aux_in_eval):
            branch = getattr(self, f'debranch{int(d) + 1}')
            aux_out = branch([e[0] for e in enc] + [dec4], [(e[1], e[2]) for e in enc], img_size)
        if out_feat:
            return {'seg': [out, aux_out], 'feat': enc[3][0].mean(dim=1)}
        return [out, aux_out]


class BASE_DSN(MDViT_DSN):
    """Drop-in for Models.Transformer.base.BASE_DSN (base.py:515-696): BASE with domain-specific norms — the MDViT_DSN trunk
    without auxiliary branches; forward(x, domain_label, d) returns the main logits only (base.py:651-693)."""

    def __init__(self, img_size=512, in_chans=3, num_stages=4, num_layers=[2, 2, 2, 2], embed_dims=[64, 128, 320, 512],
                 mlp_ratios=[8, 8, 4, 4], num_heads=[8, 8, 8, 8], qkv_bias=True, qk_scale=None, drop_rate=0., attn_drop_rate=0.,
                 drop_path_rate=0.0, norm_layer=partial(nn.LayerNorm, eps=1e-6), conv_norm=nn.BatchNorm2d, adapt_method=None,
                 num_domains=4, feature_dim=512, **kwargs):
        super().__init__(img_size, in_chans, num_stages, num_layers, embed_dims, mlp_ratios, num_heads, qkv_bias, qk_scale, drop_rate,
                         attn_drop_rate, drop_path_rate, norm_layer, conv_norm, adapt_method, num_domains, decoder_name=None)

    def forward(self, x, domain_label=None, d=None, out_feat=False, out_seg=True):
        img_size = x.shape[2:]
        int(d)      # base.py:230-280,672: the norm lists are indexed with int(d)
        enc = self._trunk_forward(x, domain_label, d)
        if not out_seg:
            return {'seg': None, 'feat': enc[3][0].mean(dim=1)}
        dec4, h, w = self._decode(enc, domain_label, d)
        out = self._head(dec4, h, w, img_size)
        if out_feat:
            return {'seg': out, 'feat': enc[3][0].mean(dim=1)}      # (pooled, base.py:688-690 — unlike BASE.forward)
        return out


class BASE(_Trunk):
    """Drop-in for Models.Transformer.base.BASE (base.py:340-512): MDViT without auxiliary branches."""

    def forward_multi(self, x, domain_label, domains):
        """The G single-domain forwards of one training step (multi_train_BASE.py calls forward once per domain) as ONE pass over the
        stacked batch, BatchNorm evaluated per group of B samples exactly as G separate forwards would (see MDViT.forward_multi).
        Returns [(out_d, None)] per domain."""
        G = len(domains)
        if x.shape[0] % G:
            raise ValueError("forward_multi needs G equal mini-batches stacked along dim 0")
        img_size = x.shape[2:]
        with ops.bn_groups(G if self.training else 1):
            enc = self._trunk_forward(x, domain_label)
            dec4, h, w = self._decode(enc, domain_label)
        out = self._head(dec4, h, w, img_size)
        return [(o, None) for o in ops.SplitDomainsFn.apply(out, G)]

    def __init__(self, img_size=512, in_chans=3, num_stages=4, num_layers=[2, 2, 2, 2], embed_dims=[64, 128, 320, 512],
                 mlp_ratios=[8, 8, 4, 4], num_heads=[8, 8, 8, 8], qkv_bias=True, qk_scale=None, drop_rate=0., attn_drop_rate=0.,
                 drop_path_rate=0.0, norm_layer=partial(nn.LayerNorm, eps=1e-6), conv_norm=nn.BatchNorm2d, adapt_method=None,
                 num_domains=4, **kwargs):
        super().__init__()
        if qk_scale is not None:
            raise ValueError("mdvit_b200 implements qk_scale=None")
        self._build_trunk(in_chans, num_stages, num_layers, embed_dims, mlp_ratios, num_heads, qkv_bias, drop_rate, attn_drop_rate,
                          drop_path_rate, norm_layer, conv_norm, adapt_method, num_domains, label_only_guard=True)
        self.apply(self._init_weights)

    def forward(self, x, domain_label=None, out_feat=False, out_seg=True):
        img_size = x.shape[2:]
        enc = self._trunk_forward(x, domain_label)
        if not out_seg:
            return {'seg': None, 'feat': enc[3][0].mean(dim=1)}
        dec4, h, w = self._decode(enc, domain_label)
        out = self._head(dec4, h, w, img_size)
        if out_feat:
            # base.py:509-510 returns the un-pooled last encoder map [B, C, H/32, W/32] here (only out_seg=False pools)
            t3, H3, W3 = enc[3]
            return {'seg': out, 'feat': t3.transpose(1, 2).reshape(t3.shape[0], t3.shape[2], H3, W3).contiguous()}
        return out
