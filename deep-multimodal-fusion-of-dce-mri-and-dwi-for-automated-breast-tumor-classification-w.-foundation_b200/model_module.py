"""B200-native drop-in for the reference's ``model_module`` (DWI / DCE encoders + late fusion).

Same class names, constructor arguments, parameter names / shapes (``state_dict`` compatible,
so checkpoints and the reference's name-based optimiser grouping keep working) and the
same ``forward`` contracts as /root/reference/code/model_module.py:

    ModelMaskHeadBackbone(method, parameters_dict, backbone=None).forward(x, masks=None)
        -> (logits[B,K], aux, mask_pred[B,1,32,32])                    (reference :481-733)
    FusionModel(parameters_dict).forward(raw_feats_dwi, raw_feats_dce, dwi_mask_pred, dce_mask_pred)
        -> (logits[B,K], fused_mask_logits[B,1,32,32], aux)            (reference :821-1000)

The sub-modules are parameter containers; the arithmetic of an eval-mode forward runs in
the hand-written sm_100a kernels behind include/b200_fusion.h (tcgen05/TMEM implicit-GEMM
convolutions fed by TMA, SIMT kernels for the K<64 / N=1 / per-case pieces).  Activations
live in HBM as NHWC bf16; the feature maps handed back in ``aux`` are zero-copy NCHW-shaped
(channels_last) bf16 views of those buffers, 1-channel maps / gates / logits are fp32.

There is no CPU or PyTorch fallback: a forward on a non-CUDA tensor, or without the
compiled library, raises.  In training mode (`.train()`) the forward runs train_graph's
train-mode arithmetic (batch-statistic BatchNorm with running-statistics update, dropout) and
returns tensors that carry a torch-autograd node: `loss.backward()` runs the explicit backward
pass on the training kernels (CNN encoder configuration; see train_graph.py).
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch
import torch.nn as nn
from torch.nn import init

import b200_native as nat

__all__ = [
    "FeatureSpec", "SEBlock", "TemporalAttention", "ChannelAttention", "MaskGuidedSpatialAttention", "ReconHead",
    "MaskHeadResize", "ResNetLiteBlock_withRecon", "Projector", "ClassificationHead", "FeatureDownAlign",
    "BackboneAdapter", "ModelMaskHeadBackbone", "GatingAttention", "FusionReduce", "CrossAttentionBlock",
    "FusionModel", "init_parameter", "initialize_model", "smooth_l1_loss",
]


def smooth_l1_loss(a, b):
    return torch.nn.functional.smooth_l1_loss(a, b)


@dataclass
class FeatureSpec:
    channels: int
    stride: int


def _only_2d(dim):
    if dim != 2:
        raise NotImplementedError("the B200 path covers dim=2 only (all BASELINE configs are 2-D)")


def _container_only(name):
    raise NotImplementedError(
        f"{name} is a parameter container in the B200 build; its arithmetic runs inside "
        "ModelMaskHeadBackbone.forward / FusionModel.forward")


def _standalone_eval(mod, name):
    """Stand-alone sub-module forwards run the eval-mode kernels (folded BatchNorm, no dropout); in training mode the
    sub-modules are driven through their parent's train-mode forward (train_graph)."""
    if mod.training:
        raise NotImplementedError(f"{name}.forward in training mode: call the parent model (ModelMaskHeadBackbone / "
                                  "FusionModel) in train mode, or .eval() for the stand-alone inference forward")


# --------------------------------------------------------------------------------------
# parameter containers (names mirror the reference so state_dict keys are identical)
# --------------------------------------------------------------------------------------
class SEBlock(nn.Module):
    """Squeeze-excite: keys fc.1.*, fc.3.* (reference :25-43)."""

    def __init__(self, channels, reduction=2, dim=2):
        super().__init__()
        _only_2d(dim)
        mid = max(channels // reduction, 1)
        self.fc = nn.Sequential(nn.AdaptiveAvgPool2d(1), nn.Conv2d(channels, mid, 1), nn.GELU(),
                                nn.Conv2d(mid, channels, 1), nn.Sigmoid())

    def forward(self, x):
        """x [B,C,H,W] -> (x * w, w [B,C,1,1]) (reference :41-43) on b200_channel_sums / b200_se_gate / b200_scale_map."""
        _standalone_eval(self, "SEBlock")
        xm = _as_nhwc_bf16(x)
        B, H, W, C = xm.shape
        se = _se_pack(self, xm.device)
        gate = torch.empty((B, C), dtype=torch.float32, device=xm.device)
        nat.se_gate(nat.channel_sums(xm), H * W, se["w1t"], se["b1"], se["w2t"], se["b2"], gate)
        y = torch.empty_like(xm)
        nat.scale_map(xm, y, gate=gate)
        return _nchw(y), gate.view(B, C, 1, 1)


class TemporalAttention(SEBlock):
    pass


class ChannelAttention(SEBlock):
    pass


class MaskGuidedSpatialAttention(nn.Module):
    """keys gamma, mask_processor.{0,1,3}.* (reference :49-97)."""

    def __init__(self, in_channels_img, in_channels_mask, hidden_channels=16, dim=2):
        super().__init__()
        _only_2d(dim)
        self.dim = dim
        self.interp_mode = "bilinear"
        self.gamma = nn.Parameter(torch.tensor(0.1))
        self.mask_processor = nn.Sequential(
            nn.Conv2d(in_channels_mask, hidden_channels, 1, bias=False), nn.GroupNorm(1, hidden_channels), nn.GELU(),
            nn.Conv2d(hidden_channels, 1, 1), nn.Sigmoid())

    def forward(self, img_features, mask_features):
        """(img [B,C,H,W], mask logits [B,1,h,w]) -> (img * (1 + gamma * A), A [B,1,H,W]) (reference :75-97)."""
        _standalone_eval(self, "MaskGuidedSpatialAttention")
        f = _as_nhwc_bf16(img_features)
        B, H, W, _ = f.shape
        dev = f.device
        m = mask_features.contiguous().float()
        if m.shape[-2:] != (H, W):
            up = torch.empty((B, 1, H, W), dtype=torch.float32, device=dev)
            nat.resize_bilinear_c1(m.view(B, *m.shape[-2:]), up.view(B, H, W))
            m = up
        mp = self.mask_processor
        attn = torch.empty((B, 1, H, W), dtype=torch.float32, device=dev)
        nat.mask_attention(m, (mp[0].out_channels, _f32(mp[0].weight.flatten(), dev), _f32(mp[1].weight, dev),
                               _f32(mp[1].bias, dev), _f32(mp[3].weight.flatten(), dev), _f32(mp[3].bias, dev), mp[1].eps), attn)
        y = torch.empty_like(f)
        nat.scale_map(f, y, attn=attn, gamma=_f32(self.gamma, dev).reshape(1))
        return _nchw(y), attn


class ReconHead(nn.Module):
    """keys conv.{0,1,3}.* (reference :100-125)."""

    def __init__(self, in_ch, recon_ch=1, upsample=False, dim=2):
        super().__init__()
        _only_2d(dim)
        self.upsample, self.dim = upsample, dim
        self.conv = nn.Sequential(nn.Conv2d(in_ch, in_ch, 3, padding=1, bias=False), nn.BatchNorm2d(in_ch), nn.GELU(),
                                  nn.Conv2d(in_ch, recon_ch, 3, padding=1))

    def forward(self, x):
        """x [B,C,H,W] -> reconstruction [B,1,H,W] fp32 (reference :113-125; recon_ch = 1, no up-sampling)."""
        _standalone_eval(self, "ReconHead")
        if self.upsample:
            raise NotImplementedError("ReconHead(upsample=True) (unused by the reference models)")
        xm = _as_nhwc_bf16(x)
        return _recon(_recon_pack(self, xm.device), xm).unsqueeze(1)


class MaskHeadResize(nn.Module):
    """keys pre.*, down_{64,128,256,512}_to_32.*, out.* (reference :131-215)."""

    def __init__(self, in_ch, mid_ch=64, out_ch=1, out_size=32, dim=2):
        super().__init__()
        _only_2d(dim)
        self.dim, self.out_size, self.interp_mode = dim, out_size, "bilinear"
        self.pre = nn.Conv2d(in_ch, mid_ch, 1)

        def chain(n):
            layers = []
            for _ in range(n):
                layers += [nn.Conv2d(mid_ch, mid_ch, 3, stride=2, padding=1), nn.GELU()]
            return nn.Sequential(*layers)

        self.down_64_to_32, self.down_128_to_32 = chain(1), chain(2)
        self.down_256_to_32, self.down_512_to_32 = chain(3), chain(4)
        self.out = nn.Conv2d(mid_ch, out_ch, 1)

    def forward(self, x):
        """x [B,C,H,W] -> mask logits [B,1,out,out] fp32 (reference :197-215)."""
        _standalone_eval(self, "MaskHeadResize")
        xm = _as_nhwc_bf16(x)
        dev = xm.device
        mk = {"pre_w": _conv_w_bf16(self.pre, dev), "pre_b": _f32(self.pre.bias, dev), "down": _mask_down_pack(self, dev),
              "out_w": _f32(self.out.weight.flatten(), dev), "out_b_host": float(self.out.bias.detach().float().cpu().item())}
        return _mask_head(mk, xm, self.out_size)


class ResNetLiteBlock_withRecon(nn.Module):
    """keys bottlenecks.N.{0,1,4,5,7,8}.*, skip.{0,1}.*, se.*, reconstruct.* (reference :220-316)."""

    def __init__(self, in_ch, out_ch, downsample=False, recon_ch=1, use_se=False, se_reduction=2, dropout=0.4, dim=2,
                 num_repeats=1, downsample_each_repeat=False, mid_squeeze=2):
        super().__init__()
        _only_2d(dim)
        self.dim, self.num_repeats = dim, num_repeats
        self.stride = 2 if downsample else 1
        self.downsample_each_repeat = downsample_each_repeat
        mid = max(out_ch // mid_squeeze, 1)
        self.bottlenecks = nn.ModuleList()
        for i in range(num_repeats):
            s = self.stride if (i == 0 or downsample_each_repeat) else 1
            self.bottlenecks.append(nn.Sequential(
                nn.Conv2d(in_ch if i == 0 else out_ch, mid, 1, stride=s, bias=False), nn.BatchNorm2d(mid), nn.GELU(),
                nn.Dropout(p=dropout),
                nn.Conv2d(mid, mid, 3, padding=1, bias=False), nn.BatchNorm2d(mid), nn.GELU(),
                nn.Conv2d(mid, out_ch, 1, bias=False), nn.BatchNorm2d(out_ch)))
        self.act = nn.GELU()
        self.dropout = nn.Dropout(p=dropout)
        if self.stride > 1 or in_ch != out_ch:
            self.skip = nn.Sequential(nn.Conv2d(in_ch, out_ch, 1, stride=self.stride, bias=False),
                                      nn.BatchNorm2d(out_ch))
        else:
            self.skip = None
        self.use_se = use_se
        self.se = SEBlock(out_ch, reduction=se_reduction, dim=dim) if use_se else None
        self.recon_ch = int(recon_ch)
        self.reconstruct = ReconHead(out_ch, recon_ch, upsample=False, dim=dim) if self.recon_ch > 0 else None

    def forward(self, x):
        """x [B,Cin,H,W] (Cin a multiple of 64) -> (out [B,Cout,H/s,W/s], recon [B,1,H/s,W/s] | None) (reference :298-316)."""
        _standalone_eval(self, "ResNetLiteBlock_withRecon")
        xm = _as_nhwc_bf16(x)
        if xm.shape[-1] % 64:
            raise NotImplementedError("stand-alone block forward needs >= 64 input channels (block1 reads the raw input "
                                      "through the encoder's fused stem)")
        dev = xm.device
        pk = _block_pack(self, dev)
        pk["stride"], pk["downsample_each_repeat"] = self.stride, bool(self.downsample_each_repeat) and len(self.bottlenecks) > 1
        for bt in pk["bott"]:
            bt["w0"] = _conv_w_bf16(bt["conv0"], dev)
        st = self.stride
        b0 = pk["bott"][0]
        if "skip" in pk:
            skip = nat.conv_gemm(xm, _conv_w_bf16(pk["skip"]["conv"], dev), taps=1, scale=pk["skip"]["s"], bias=pk["skip"]["b"],
                                 stride=st)
        else:
            skip = xm
        mid = nat.conv_gemm(xm, b0["w0"], taps=1, scale=b0["s1"], bias=b0["b1"], act=1, stride=st)
        host = ModelMaskHeadBackbone.__new__(ModelMaskHeadBackbone)
        host._drop = None
        out, rec, _, _ = ModelMaskHeadBackbone._run_block(host, pk, mid, skip, True)
        return _nchw(out), (rec.unsqueeze(1) if rec is not None else None)


class Projector(nn.Module):
    """keys proj.{0,1,3,4}.* (reference :323-348)."""

    def __init__(self, in_ch, proj_dim=64, dim=2):
        super().__init__()
        _only_2d(dim)
        self.dim = dim
        self.proj = nn.Sequential(nn.Conv2d(in_ch, proj_dim, 1, bias=False), nn.BatchNorm2d(proj_dim), nn.GELU(),
                                  nn.Conv2d(proj_dim, proj_dim, 1, bias=False), nn.BatchNorm2d(proj_dim), nn.GELU())

    def forward(self, x):
        """x [B,C,H,W] (C >= 64, or a 1-channel fp32 map) -> [B,proj_dim,H,W] (reference :346-348)."""
        _standalone_eval(self, "Projector")
        if x.shape[1] == 1:
            src = x[:, 0].contiguous().float()
            pp = _proj_pack(self, src.device)
            g = torch.empty((*src.shape, pp["w0_vec"].numel()), dtype=torch.bfloat16, device=src.device)
            nat.lift_c1(src, pp["w0_vec"], pp["s0"], pp["b0"], g)
        else:
            xm = _as_nhwc_bf16(x)
            pp = _proj_pack(self, xm.device)
            g = nat.conv_gemm(xm, pp["w0"], taps=1, scale=pp["s0"], bias=pp["b0"], act=1)
        return _nchw(nat.conv_gemm(g, pp["w3"], taps=1, scale=pp["s3"], bias=pp["b3"], act=1))


class ClassificationHead(nn.Module):
    """keys fc.* (reference :355-369)."""

    def __init__(self, in_ch, num_classes, dim=2, normalize=True):
        super().__init__()
        _only_2d(dim)
        self.pool, self.flatten = nn.AdaptiveAvgPool2d((1, 1)), nn.Flatten()
        self.fc = nn.Linear(in_ch, num_classes)
        self.normalize = normalize

    def forward(self, x):
        """x [B,C,H,W] -> logits [B,K] fp32: GAP, L2-normalise, Linear (reference :364-369)."""
        _standalone_eval(self, "ClassificationHead")
        xm = _as_nhwc_bf16(x)
        B, H, W, _ = xm.shape
        logits = torch.empty((B, self.fc.out_features), dtype=torch.float32, device=xm.device)
        nat.cls_head(nat.channel_sums(xm), None, H * W, _f32(self.fc.weight, xm.device), _f32(self.fc.bias, xm.device),
                     self.normalize, logits)
        return logits


class FeatureDownAlign(nn.Module):
    """keys proj.{0,1}.* (reference :371-396)."""

    def __init__(self, in_ch, out_ch, dim=2, downsample=True):
        super().__init__()
        _only_2d(dim)
        self.downsample = downsample
        if in_ch != out_ch or downsample:
            k, s, p = (3, 2, 1) if downsample else (1, 1, 0)
            self.proj = nn.Sequential(nn.Conv2d(in_ch, out_ch, k, stride=s, padding=p, bias=False),
                                      nn.BatchNorm2d(out_ch), nn.GELU())
        else:
            self.proj = nn.Identity()

    def forward(self, x):
        """x [B,Cin,H,W] -> conv + BN + GELU (1x1, or 3x3 stride 2 when `downsample`) (reference :393-396)."""
        _standalone_eval(self, "FeatureDownAlign")
        if isinstance(self.proj, nn.Identity):
            return x
        xm = _as_nhwc_bf16(x)
        s, b = _bn_fold(self.proj[1], xm.device)
        taps, st = (9, 2) if self.downsample else (1, 1)
        return _nchw(nat.conv_gemm(xm, _conv_w_bf16(self.proj[0], xm.device), taps=taps, scale=s, bias=b, act=1, stride=st))


class _DynamoDisabled(nn.Module):
    """Stands in for the wrapper `torch._dynamo.disable(backbone)` returns (reference :539): the wrapped module
    sits under `_orig_mod`, which is what puts `backbone._orig_mod.*` / `backbone_adapter.backbone._orig_mod.*`
    keys into the reference's checkpoints.  Everything else is forwarded to the wrapped module."""

    def __init__(self, module):
        super().__init__()
        self._orig_mod = module

    def forward(self, *args, **kwargs):
        return self._orig_mod(*args, **kwargs)

    def __getattr__(self, name):
        try:
            return super().__getattr__(name)
        except AttributeError:
            return getattr(self._modules["_orig_mod"], name)


class BackboneAdapter(nn.Module):
    """keys backbone.*, necks.f{1,2,3}.{0,1,3,4}.* (reference :401-476)."""

    def __init__(self, backbone, selected_indices_chains, out_channels=(64, 128, 256), dim=2, is_transformer=False):
        super().__init__()
        _only_2d(dim)
        assert len(selected_indices_chains) == 3, "Must provide 3 chains for f1/f2/f3"
        assert len(out_channels) == 3, "Must provide 3 output channels for f1/f2/f3"
        self.backbone = backbone
        self.selected_indices_chains = selected_indices_chains
        self.dim, self.is_transformer = dim, is_transformer
        info = backbone.feature_info
        self.features = [FeatureSpec(c, s) for c, s in zip(info.channels(), info.reduction())]
        self.necks = nn.ModuleDict()
        for i, chain in enumerate(selected_indices_chains):
            cin, cout = sum(self.features[j].channels for j in chain), out_channels[i]
            self.necks[f"f{i + 1}"] = nn.Sequential(
                nn.Conv2d(cin, cout, 3, padding=1), nn.BatchNorm2d(cout), nn.GELU(),
                nn.Conv2d(cout, cout, 3, padding=1), nn.BatchNorm2d(cout), nn.GELU())

    def forward(self, x):
        """x [B,C,H,W] normalised input -> (f1_b, f2_b, f3_b) (reference :449-476): backbone chains + the two 3x3
        conv + BN + GELU necks."""
        _standalone_eval(self, "BackboneAdapter")
        if not hasattr(self.backbone, "forward_chains"):
            raise NotImplementedError("BackboneAdapter needs a backbone from foundation_model.build_medical_backbone")
        dev = x.device
        outs = []
        for i, cat in enumerate(self.backbone.forward_chains(x.contiguous().float(), self.selected_indices_chains, None)):
            nk = self.necks[f"f{i + 1}"]
            s0, b0 = _bn_fold(nk[1], dev, nk[0].bias)
            s3, b3 = _bn_fold(nk[4], dev, nk[3].bias)
            t = nat.conv_gemm(cat, _conv_w_bf16(nk[0], dev), taps=9, scale=s0, bias=b0, act=1)
            outs.append(_nchw(nat.conv_gemm(t, _conv_w_bf16(nk[3], dev), taps=9, scale=s3, bias=b3, act=1)))
        return tuple(outs)


class GatingAttention(nn.Module):
    """keys fc.* (reference :745-780)."""

    def __init__(self, feat_dim, use_mask_attention=True, dim=2):
        super().__init__()
        self.use_mask_attention, self.dim = use_mask_attention, dim
        self.fc = nn.Linear(feat_dim * 2 + (2 if use_mask_attention else 0), 2)

    def forward(self, pvec_dwi, pvec_dce, dwi_mask=None, dce_mask=None):
        """pooled vectors [B,C] (+ encoder mask logits) -> softmax gating weights [B,2] (reference :758-780)."""
        pd_, pc_ = pvec_dwi.contiguous().float(), pvec_dce.contiguous().float()
        if not pd_.is_cuda:
            raise nat.B200NativeError("GatingAttention.forward needs CUDA tensors (no CPU path)")
        B, C = pd_.shape
        use = self.use_mask_attention and dwi_mask is not None and dce_mask is not None
        md = dwi_mask.contiguous().float() if use else None
        mc = dce_mask.contiguous().float() if use else None
        D = 2 * C + (2 if use else 0)
        if self.fc.in_features != D:
            raise RuntimeError("GatingAttention: the Linear expects the mask confidences it was built with")
        gx = torch.empty((B, D), dtype=torch.float32, device=pd_.device)
        alpha = torch.empty((B, 2), dtype=torch.float32, device=pd_.device)
        nat._call("b200_gating_fwd", None, nat._ptr(pd_), nat._ptr(pc_), B, C, 1, nat._ptr(md), nat._ptr(mc),
                  md[0].numel() if use else 0, nat._ptr(_f32(self.fc.weight, pd_.device)), nat._ptr(_f32(self.fc.bias, pd_.device)),
                  nat._ptr(gx), nat._ptr(alpha), nat._stream())
        return alpha


class FusionReduce(nn.Module):
    """keys reduce.{0,1}.* (reference :782-794)."""

    def __init__(self, in_ch, out_ch, dim=2):
        super().__init__()
        _only_2d(dim)
        self.reduce = nn.Sequential(nn.Conv2d(in_ch, out_ch, 1, bias=False), nn.BatchNorm2d(out_ch), nn.GELU())

    def forward(self, x):
        """x [B,2C,H,W] -> 1x1 conv + BN + GELU (reference :793-794)."""
        _standalone_eval(self, "FusionReduce")
        xm = _as_nhwc_bf16(x)
        s, b = _bn_fold(self.reduce[1], xm.device)
        return _nchw(nat.conv_gemm(xm, _conv_w_bf16(self.reduce[0], xm.device), taps=1, scale=s, bias=b, act=1))


class CrossAttentionBlock(nn.Module):
    """keys cross_attn.*, attn_ffn.{0,1,3}.* (reference :799-818)."""

    def __init__(self, channels, num_heads=4):
        super().__init__()
        self.cross_attn = nn.MultiheadAttention(embed_dim=channels, num_heads=num_heads, batch_first=True)
        self.attn_ffn = nn.Sequential(nn.LayerNorm(channels), nn.Linear(channels, channels), nn.GELU(),
                                      nn.Linear(channels, channels))

    def forward(self, query_tokens, key_value_tokens):
        """(q tokens [B,T,C], kv tokens [B,T,C]) -> (attn_out + FFN(attn_out) [B,T,C], head-averaged weights [B,T,T])
        (reference :814-818) on the fp32 token kernels (b200_sgemm / b200_mha_fwd / b200_ln_fwd)."""
        q_, kv_ = query_tokens.contiguous().float(), key_value_tokens.contiguous().float()
        if not q_.is_cuda:
            raise nat.B200NativeError("CrossAttentionBlock.forward needs CUDA tensors (no CPU path)")
        B, T, C = q_.shape
        dev, R, NH = q_.device, B * T, self.cross_attn.num_heads
        z = lambda *sh: torch.empty(sh, dtype=torch.float32, device=dev)
        Win, b_in = _f32(self.cross_attn.in_proj_weight, dev), _f32(self.cross_attn.in_proj_bias, dev)
        Q, KV, P, CTX, AO, LN, G1, LOW = z(R, C), z(R, 2 * C), z(B, NH, T, T), z(R, C), z(R, C), z(R, C), z(R, C), z(R, C)
        nat.sgemm(q_.view(R, C), Win[:C], Q, trans_b=True, bias=b_in[:C])
        nat.sgemm(kv_.view(R, C), Win[C:], KV, trans_b=True, bias=b_in[C:])
        nat.mha_fwd(Q, KV[:, :C], KV[:, C:], B, NH, P, CTX)
        nat.sgemm(CTX, _f32(self.cross_attn.out_proj.weight, dev), AO, trans_b=True, bias=_f32(self.cross_attn.out_proj.bias, dev))
        ln = self.attn_ffn[0]
        nat.ln_fwd(AO, _f32(ln.weight, dev), _f32(ln.bias, dev), ln.eps, LN, z(R), z(R))
        nat.sgemm(LN, _f32(self.attn_ffn[1].weight, dev), G1, trans_b=True, bias=_f32(self.attn_ffn[1].bias, dev), act=1)
        nat.sgemm(G1, _f32(self.attn_ffn[3].weight, dev), LOW, trans_b=True, bias=_f32(self.attn_ffn[3].bias, dev), res=AO)
        return LOW.view(B, T, C), P.mean(dim=1)


# --------------------------------------------------------------------------------------
# weight packing helpers (one-off layout transforms; not on the per-batch path)
# --------------------------------------------------------------------------------------
def _f32(t, dev):
    return t.detach().to(device=dev, dtype=torch.float32).contiguous()


def _conv_w_bf16(conv, dev):
    """[Cout,Cin,kh,kw] -> [Cout, kh*kw*Cin] bf16 (k = tap*Cin + c)."""
    w = conv.weight.detach().to(dev)
    return w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).to(torch.bfloat16).contiguous()


def _bn_fold(bn, dev, conv_bias=None):
    """Eval-mode BatchNorm as a per-channel affine; a preceding conv bias folds into the shift."""
    g, b = _f32(bn.weight, dev), _f32(bn.bias, dev)
    m, v = _f32(bn.running_mean, dev), _f32(bn.running_var, dev)
    scale = g / torch.sqrt(v + bn.eps)
    shift = b - m * scale
    if conv_bias is not None:
        shift = shift + _f32(conv_bias, dev) * scale
    return scale.contiguous(), shift.contiguous()


def _se_pack(se, dev):
    c1, c2 = se.fc[1], se.fc[3]
    return {"w1": _f32(c1.weight.flatten(1), dev), "b1": _f32(c1.bias, dev),
            "w2": _f32(c2.weight.flatten(1), dev), "b2": _f32(c2.bias, dev),
            "w1t": _f32(c1.weight.flatten(1).t(), dev), "w2t": _f32(c2.weight.flatten(1).t(), dev)}


def _recon_pack(rh, dev):
    s, b = _bn_fold(rh.conv[1], dev)
    w3 = rh.conv[3].weight.detach().to(dev)  # [1,C,3,3]
    if w3.shape[0] != 1:
        raise NotImplementedError("reconstruction heads with recon_ch != 1")
    return {"w0": _conv_w_bf16(rh.conv[0], dev), "s0": s, "b0": b,
            "w3": w3[0].permute(1, 2, 0).reshape(9, -1).float().contiguous(), "b3": _f32(rh.conv[3].bias, dev)}


def _proj_pack(pr, dev):
    s0, b0 = _bn_fold(pr.proj[1], dev)
    s3, b3 = _bn_fold(pr.proj[4], dev)
    p = {"s0": s0, "b0": b0, "w3": _conv_w_bf16(pr.proj[3], dev), "s3": s3, "b3": b3}
    if pr.proj[0].in_channels == 1:
        p["w0_vec"] = _f32(pr.proj[0].weight.flatten(), dev)
    else:
        p["w0"] = _conv_w_bf16(pr.proj[0], dev)
    return p


def _mask_down_pack(mh, dev):
    """MaskHeadResize's strided stacks (reference :153-181): map size -> [(weight [64, 9*64] bf16, bias)] of its
    3x3 / stride-2 convs (each followed by GELU)."""
    out = {}
    for size, name in ((64, "down_64_to_32"), (128, "down_128_to_32"), (256, "down_256_to_32"), (512, "down_512_to_32")):
        seq = getattr(mh, name, None)
        if seq is not None:
            out[size] = [(_conv_w_bf16(m, dev), _f32(m.bias, dev)) for m in seq if isinstance(m, nn.Conv2d)]
    return out


def _mask_head(mk, m_in, mask_size):
    """MaskHeadResize.forward (reference :197-215) on an NHWC bf16 map -> mask logits [B,1,S,S] fp32 at the
    head's output size and, when the `pre` map is not resized (32 x 32 input), nothing else.  The final 1x1
    `out` conv (64 -> 1) always runs as an fp32 dot product inside the epilogue of the GEMM before it."""
    B, H, W, _ = m_in.shape
    dev = m_in.device
    out_w, out_b = mk["out_w"].view(1, -1), mk["out_b_host"]
    if H == mask_size or H not in mk["down"]:
        # identity path, or the bilinear fallback (:205-211): resize and the 1x1 `out` conv are both linear and the
        # resize acts per channel, so the 1-channel logits are resized instead of the 64-channel map
        small = torch.empty((B, 1, H, W), dtype=torch.float32, device=dev)
        nat.conv_gemm(m_in, mk["pre_w"], taps=1, bias=mk["pre_b"], store=False, dot_w=out_w, dot_out=small, dot_bias=out_b)
        if H == mask_size:
            return small
        mask = torch.empty((B, 1, mask_size, mask_size), dtype=torch.float32, device=dev)
        nat.resize_bilinear_c1(small.view(B, H, W), mask.view(B, mask_size, mask_size))
        return mask
    # strided stacks: pre (1x1, bias) -> [3x3 stride 2 + GELU] x n -> out
    t = nat.conv_gemm(m_in, mk["pre_w"], taps=1, bias=mk["pre_b"])
    stack = mk["down"][H]
    for w, b in stack[:-1]:
        t = nat.conv_gemm(t, w, taps=9, bias=b, act=1, stride=2)
    w, b = stack[-1]
    S = t.shape[1] // 2
    mask = torch.empty((B, 1, S, S), dtype=torch.float32, device=dev)
    nat.conv_gemm(t, w, taps=9, bias=b, act=1, stride=2, store=False, dot_w=out_w, dot_out=mask, dot_bias=out_b)
    return mask


def _block_pack(blk, dev):
    p = {"bott": []}
    for bt in blk.bottlenecks:
        s1, b1 = _bn_fold(bt[1], dev)
        s5, b5 = _bn_fold(bt[5], dev)
        s8, b8 = _bn_fold(bt[8], dev)
        p["bott"].append({"conv0": bt[0], "s1": s1, "b1": b1, "w4": _conv_w_bf16(bt[4], dev), "s5": s5, "b5": b5,
                          "w7": _conv_w_bf16(bt[7], dev), "s8": s8, "b8": b8,
                          "conv7_f32": bt[7].weight.detach().to(dev).flatten(1).float()})
    if blk.skip is not None:
        ss, sb = _bn_fold(blk.skip[1], dev)
        p["skip"] = {"conv": blk.skip[0], "s": ss, "b": sb}
    if blk.se is not None:
        p["se"] = _se_pack(blk.se, dev)
    if blk.reconstruct is not None:
        p["recon"] = _recon_pack(blk.reconstruct, dev)
    return p


def _transformer_pack(stage, out_proj, dev):
    """TransformerStage + trans_out_proj (reference transformer_model.py:137-175, model_module.py:568-579)."""
    pe = stage.patch_embed
    if pe.proj.kernel_size != (2, 2) or pe.proj.stride != (2, 2):
        raise NotImplementedError("only patch_size=2 (the reference default) is built")
    E = pe.proj.out_channels
    tr = {"E": E, "pe_w": _conv_w_bf16(pe.proj, dev), "pe_b": _f32(pe.proj.bias, dev),
          "pe_ln": (_f32(pe.norm.weight, dev), _f32(pe.norm.bias, dev), pe.norm.eps), "layers": [],
          "out_w": _conv_w_bf16(out_proj, dev), "out_b": _f32(out_proj.bias, dev)}
    for blk in stage.transformer.layers:
        at = blk.attn
        wqkv = at.qkv.weight.detach().to(dev)
        bqkv = at.qkv.bias.detach().to(dev).float() if at.qkv.bias is not None else torch.zeros(3 * E, device=dev)
        g1, g2 = _f32(blk.gamma1, dev), _f32(blk.gamma2, dev)
        tr["layers"].append({
            "heads": at.num_heads, "dh": at.head_dim,
            "ln1": (_f32(blk.norm1.weight, dev), _f32(blk.norm1.bias, dev), blk.norm1.eps),
            "ln2": (_f32(blk.norm2.weight, dev), _f32(blk.norm2.bias, dev), blk.norm2.eps),
            "wqkv": wqkv.to(torch.bfloat16).contiguous(), "bqkv": bqkv.contiguous(),
            # x + gamma * (W y + b)  ==  (acc * gamma + gamma * b) + x : LayerScale folds into the epilogue affine
            "wproj": at.proj.weight.detach().to(dev, torch.bfloat16).contiguous(), "sproj": g1,
            "bproj": (g1 * _f32(at.proj.bias, dev)).contiguous(),
            "wfc1": blk.mlp.fc1.weight.detach().to(dev, torch.bfloat16).contiguous(), "bfc1": _f32(blk.mlp.fc1.bias, dev),
            "wfc2": blk.mlp.fc2.weight.detach().to(dev, torch.bfloat16).contiguous(), "sfc2": g2,
            "bfc2": (g2 * _f32(blk.mlp.fc2.bias, dev)).contiguous(),
            # the block's nn.Dropout modules, read at every forward: MC-dropout inference switches them per module
            "attn_drop": at.attn_drop, "proj_drop": at.proj_drop, "mlp_drop": blk.mlp.drop,
        })
    return tr


def _transformer_dropouts(tr):
    """True when some nn.Dropout of the packed transformer stage is in train mode with p > 0 (MC dropout)."""
    return any(m.training and m.p > 0 for ly in tr["layers"] for m in (ly["attn_drop"], ly["proj_drop"], ly["mlp_drop"]))


def _transformer_stage(tr, x, drop=None):
    """x [B,H,W,C] bf16 NHWC -> (f3 [B,H/2,W/2,c3] bf16, per-case channel sums of f3).

    `drop(segments, p)` (the encoder's per-launch seed stream, MC-dropout inference) -> (p, seed, segments): every
    nn.Dropout of a block that is in train mode with p > 0 applies inside the launch it follows, timm's placement
    (DESIGN.md section 2): attn_drop on the softmax probabilities, proj_drop on proj(o) before LayerScale and the
    residual, mlp.drop after the GELU and again on fc2's output before LayerScale and the residual.

    Pre-norm blocks exactly as transformer_model.py:68-133 (eval: dropout is identity).  The patch embedding is a
    2x2/stride-2 implicit GEMM and qkv / proj / fc1 / fc2 run on the tcgen05 GEMM kernel, with LayerScale + residual
    folded into the proj / fc2 epilogues.  Attention is one b200_attention launch per block: S = Q K^T per
    (case, head) in TMEM, the softmax in registers, and P V straight off the packed qkv rows."""
    B, H, W, _ = x.shape
    E = tr["E"]
    dev = x.device
    tok = nat.conv_gemm(x, tr["pe_w"], taps=4, bias=tr["pe_b"])  # [B, H/2, W/2, E]
    Ht, Wt = tok.shape[1], tok.shape[2]
    N = Ht * Wt
    M = B * N
    # the residual stream t is kept in fp32 across the blocks (12 bf16 roundings of it would dominate the error);
    # everything that feeds a tensor-core GEMM is bf16
    t = nat.layernorm(tok.view(M, E), *tr["pe_ln"], out_dtype=torch.float32)
    h = torch.empty((M, E), dtype=torch.bfloat16, device=dev)
    qkv = torch.empty((M, 3 * E), dtype=torch.bfloat16, device=dev)
    o = torch.empty((M, E), dtype=torch.bfloat16, device=dev)
    u = torch.empty((M, 4 * E), dtype=torch.bfloat16, device=dev)

    def dr(mod):  # (p, seed) of one launch for an active Dropout module, else None
        return drop(1, float(mod.p))[:2] if drop is not None and mod.training and mod.p > 0 else None

    for ly in tr["layers"]:
        heads, dh = ly["heads"], ly["dh"]
        nat.layernorm(t, *ly["ln1"], out=h)
        nat.linear(h, ly["wqkv"], bias=ly["bqkv"], out=qkv)
        nat.attention(qkv, o, B, N, heads, dh, dropout=dr(ly["attn_drop"]))  # transformer_model.py:101-112 in one launch
        last = ly is tr["layers"][-1]
        t2 = nat.linear_f32(o, ly["wproj"], scale=ly["sproj"], bias=ly["bproj"], res=t, res_mode=2,
                            out_dtype=torch.float32, dropout=dr(ly["proj_drop"]))
        nat.layernorm(t2, *ly["ln2"], out=h)
        nat.linear(h, ly["wfc1"], bias=ly["bfc1"], act=1, out=u, dropout=dr(ly["mlp_drop"]))
        t = nat.linear_f32(u, ly["wfc2"], scale=ly["sfc2"], bias=ly["bfc2"], res=t2, res_mode=2,
                           out_dtype=torch.bfloat16 if last else torch.float32, dropout=dr(ly["mlp_drop"]))
    c3 = tr["out_w"].shape[0]
    gap = torch.zeros((B, c3), dtype=torch.float32, device=dev)
    f3 = nat.conv_gemm(t.view(B, Ht, Wt, E), tr["out_w"], taps=1, bias=tr["out_b"], gap=gap)
    return f3, gap


def _state_signature(module):
    return tuple((t.data_ptr(), t._version) for t in list(module.parameters()) + list(module.buffers()))


class _PackedWeightsMixin:
    """Owner of a packed-weight cache (bf16 [Cout, taps*Cin] slabs, folded BatchNorm affines).  The cache key is
    (data_ptr, version) of every parameter and buffer, which in-place writes through `.data` do not change
    (init_parameter below writes that way, as the reference's does, and so do EMA / SWA swaps): every entry point that
    can rewrite weights behind the version counter drops the cache instead - `initialize_model`, `load_state_dict`,
    `_apply` (.to / .half / .cuda) - and `invalidate_packed()` is public for callers that poke `.data` themselves."""

    def invalidate_packed(self):
        self._pack_cache = None

    def _apply(self, fn, *a, **k):
        self._pack_cache = None
        return super()._apply(fn, *a, **k)

    def load_state_dict(self, *a, **k):
        self._pack_cache = None
        return super().load_state_dict(*a, **k)


def _as_nhwc_bf16(t):
    """NCHW-shaped tensor -> NHWC bf16 contiguous buffer (zero-copy for our own channels_last views)."""
    if not t.is_cuda:
        raise nat.B200NativeError("feature maps must be CUDA tensors (no CPU path)")
    v = t.permute(0, 2, 3, 1)
    if v.dtype == torch.bfloat16 and v.is_contiguous():
        return v
    return v.to(torch.bfloat16).contiguous()


def _nchw(t):
    return t.permute(0, 3, 1, 2)


def _staged_tiles(H, W):
    """True when the GEMM kernel tiles an H x W map into whole 128-pixel boxes (W divides 128 and the rows per
    tile divide H): only then can its epilogue stage tiles in shared memory, which the fused per-case channel
    sums rely on.  The 14 x 14 ViT grid does not; its pools go through b200_channel_sums."""
    return W <= 128 and 128 % W == 0 and H % (128 // W) == 0


def _conv_gap(x, w, **kw):
    """conv_gemm that also returns the per-case channel sums of its output (global average pool)."""
    B, H, W, _ = x.shape
    if _staged_tiles(H, W):
        gap = torch.zeros((B, w.shape[0]), dtype=torch.float32, device=x.device)
        return nat.conv_gemm(x, w, gap=gap, **kw), gap
    out = nat.conv_gemm(x, w, **kw)
    return out, nat.channel_sums(out)


def _recon(rc, x):
    """ReconHead (reference :113-118): 3x3 conv + BN + GELU on the tensor cores with the final 3x3, C->1
    conv folded in - the GEMM epilogue emits the 9 per-tap dot products of its result, a shift-sum finishes
    the convolution, and the intermediate C-channel map is never written to HBM."""
    B, H, W, C = x.shape
    rec = torch.empty((B, H, W), dtype=torch.float32, device=x.device)
    if C > 256:
        # the fused form needs all C output channels in one 256-wide accumulator tile; wider heads (768 on the
        # ViT path) write the intermediate map and finish with the stand-alone C->1 kernel
        t = nat.conv_gemm(x, rc["w0"], taps=9, scale=rc["s0"], bias=rc["b0"], act=1)
        return nat.conv3x3_c1(t, rc["w3"], rc["b3"], rec)
    d = torch.empty((B, H, W, 9), dtype=torch.float32, device=x.device)
    nat.conv_gemm(x, rc["w0"], taps=9, scale=rc["s0"], bias=rc["b0"], act=1, store=False, dot_w=rc["w3"], dot_out=d)
    return nat.tapsum(d, rc["b3"], rec)


# --------------------------------------------------------------------------------------
# encoder
# --------------------------------------------------------------------------------------
class ModelMaskHeadBackbone(_PackedWeightsMixin, nn.Module):
    """DWI / DCE encoder (reference :481-733).  ``aux_mode``: "full" materialises every output of
    the reference API; "logits" skips what the fusion logits do not depend on (reconstruction heads,
    projectors, the encoder's own classifier) and returns None for those entries."""

    def __init__(self, method, parameters_dict, backbone=None):
        super().__init__()
        self.method = method
        self.channel_num = parameters_dict[f"{method}_channel_num"]
        self.num_classes = parameters_dict["class_num"]
        self.dim = parameters_dict["dim"]
        _only_2d(self.dim)
        mp = parameters_dict[f"{method}_model_parameters"]
        self.enable_modality_attention = mp["enable_modality_attention"]
        self.use_se = mp["use_se"]
        self.use_hybrid_transformer = mp["use_hybrid_transformer"]
        self.use_backbone = mp["use_backbone"]
        self.channels = mp["channels"]
        self.proj_dim = mp["proj_dim"]
        self.dropout = mp["dropout"]
        self.num_repeats = mp["repeat_blocks"]
        self.mid_squeeze = mp["mid_squeeze"]
        self.downsample = mp["downsample"]
        self.downsample_each_repeat = mp["downsample_each_repeat"]
        self.selected_indices_chains = mp["backbone_index_lists"]
        self.backbone_out_channels = mp["backbone_out_channels"]
        self.transformer_backbone = mp["transformer_backbone"]
        maskp = mp["mask_parameters"]
        self.mask_enabled = maskp["mask"]
        self.mask_stage = maskp["mask_stage"].lower()
        self.mask_size = maskp["mask_target_size"][0]
        self.aux_mode = "full"
        c1, c2, c3 = self.channels

        self.proj_pool = nn.AdaptiveAvgPool2d((self.proj_dim, self.proj_dim))
        self.backbone = _DynamoDisabled(backbone) if isinstance(backbone, nn.Module) else None
        if self.use_backbone:
            self.backbone_adapter = BackboneAdapter(backbone=self.backbone, selected_indices_chains=self.selected_indices_chains,
                                                    out_channels=(c1, c1, c2), is_transformer=self.transformer_backbone)
            block1_in = c1
        else:
            block1_in = self.channel_num

        def block(cin, cout, i, recon):
            return ResNetLiteBlock_withRecon(cin, cout, downsample=self.downsample[i], recon_ch=recon,
                                             use_se=self.use_se, dim=self.dim, dropout=self.dropout,
                                             num_repeats=self.num_repeats[i],
                                             downsample_each_repeat=self.downsample_each_repeat,
                                             mid_squeeze=self.mid_squeeze)

        self.block1 = block(block1_in, c1, 0, 1)
        self.block2 = block(c1, c2, 1, 1)
        if not self.use_hybrid_transformer:
            self.block3 = block(c2, c3, 2, 0)
        else:
            from transformer_model import TransformerStage
            self.transformer = TransformerStage(in_ch=c2, embed_dim=mp["transformer_embed_dim"],
                                                depth=mp["transformer_depth"], heads=mp["transformer_heads"],
                                                patch_size=mp["transformer_patch_size"], dim=self.dim)
            self.trans_out_proj = nn.Conv2d(mp["transformer_embed_dim"], c3, kernel_size=1)

        self.modality_attention = None
        if self.enable_modality_attention:
            if method == "dce":
                self.modality_attention = TemporalAttention(self.channel_num, reduction=2)
            elif method == "dwi":
                self.modality_attention = ChannelAttention(self.channel_num, reduction=2)
            else:
                raise ValueError("Unknown method for modality attention.")
        self.f2_weight = nn.Parameter(torch.tensor(0.5))
        self.f3_weight = nn.Parameter(torch.tensor(0.5))
        self.norm_f2 = nn.GroupNorm(c1, c1)
        self.norm_f3 = nn.GroupNorm(c2, c2)
        if self.mask_enabled:
            self.f1_to_f2 = FeatureDownAlign(c1, c2, dim=self.dim, downsample=False)
            self.f2_to_f3 = FeatureDownAlign(c2, c3, dim=self.dim, downsample=False)
            mask_in = {"f1": c1, "f2": c2, "f3": c3}[self.mask_stage]
            self.mask_head = MaskHeadResize(in_ch=mask_in, out_size=self.mask_size, dim=self.dim)
            self.mask_spatial_attention = MaskGuidedSpatialAttention(in_channels_img=c3, in_channels_mask=1,
                                                                     dim=self.dim)
            if self.use_hybrid_transformer and self.mask_stage == "f3":
                raise ValueError("mask_stage='f3' not supported with hybrid transformer")
        self.classification_head = ClassificationHead(in_ch=c3, num_classes=self.num_classes, dim=self.dim)
        self.proj_f1 = Projector(c1, self.proj_dim, dim=self.dim)
        self.proj_f2 = Projector(c2, self.proj_dim, dim=self.dim)
        self.proj_r1 = Projector(1, self.proj_dim, dim=self.dim)
        self.proj_r2 = Projector(1, self.proj_dim, dim=self.dim)
        self._pack_cache = None
        self._mc_seed, self._mc_calls, self._drop = 0x5EED, 0, None

    # ------------------------------------------------------------- MC dropout ----
    def set_mc_seed(self, seed):
        """Seed of the in-kernel dropout generator (Philox, counter based): one forward consumes one seed step, so
        a fixed seed reproduces a sequence of MC passes."""
        self._mc_seed, self._mc_calls = int(seed), 0

    def _mc_dropout_p(self):
        """MC-dropout inference as the reference arms it (train_fusion.py:445-481): the module is in eval mode,
        BatchNorm frozen, but its nn.Dropout sub-modules have been put in train mode.  Returns the p of the CNN
        blocks' dropouts (0 = off); the hybrid transformer stage's own dropouts (p = 0.1) are read per module."""
        blocks = [self.block1, self.block2] + ([] if self.use_hybrid_transformer else [self.block3])
        for blk in blocks:
            for mod in blk.modules():
                if isinstance(mod, nn.Dropout) and mod.training and mod.p > 0:
                    return float(mod.p)
        return 0.0

    # ---------------------------------------------------------------- packing ----
    def _packed(self, dev):
        sig = (str(dev), _state_signature(self))
        if self._pack_cache is not None and self._pack_cache[0] == sig:
            return self._pack_cache[1]
        if self.use_backbone and not hasattr(self.backbone, "forward_chains"):
            raise NotImplementedError("use_backbone needs a backbone from foundation_model.build_medical_backbone "
                                      "(B200ViTBackbone / B200ResNetBackbone); UNI2-h is not built")
        b1 = self.block1
        if self.use_backbone:
            if self.use_hybrid_transformer or (b1.stride != 1 and b1.skip is None):
                raise NotImplementedError("backbone encoders with the hybrid transformer stage")
        elif b1.stride not in (1, 2) or b1.skip is None or self.channel_num > 32:
            raise NotImplementedError("block1 must read the raw (<=32 channel) input through a skip conv")
        blocks = {"b1": self.block1, "b2": self.block2}
        if not self.use_hybrid_transformer:
            blocks["b3"] = self.block3
        pk = {name: _block_pack(blk, dev) for name, blk in blocks.items()}
        for name, blk in blocks.items():
            pk[name]["stride"] = blk.stride
            pk[name]["downsample_each_repeat"] = bool(self.downsample_each_repeat) and len(blk.bottlenecks) > 1
            if pk[name]["downsample_each_repeat"] and blk.stride != 1:
                raise NotImplementedError("downsample_each_repeat with a strided block (the identity branch would "
                                          "not match in the reference either)")
            if blk.stride not in (1, 2) or (blk.stride == 2 and blk.skip is None):
                raise NotImplementedError("block strides other than 1 / 2")
        if self.use_hybrid_transformer:
            pk["tr"] = _transformer_pack(self.transformer, self.trans_out_proj, dev)
        if self.use_backbone:
            # necks (reference :440-447): conv bias folds into the BatchNorm shift
            pk["necks"] = []
            for i in range(3):
                nk = self.backbone_adapter.necks[f"f{i + 1}"]
                s0, b0 = _bn_fold(nk[1], dev, nk[0].bias)
                s3, b3 = _bn_fold(nk[4], dev, nk[3].bias)
                pk["necks"].append({"w0": _conv_w_bf16(nk[0], dev), "s0": s0, "b0": b0,
                                    "w3": _conv_w_bf16(nk[3], dev), "s3": s3, "b3": b3})
            pk["mix"] = {"f2": (_f32(self.f2_weight, dev).reshape(1), _f32(self.norm_f2.weight, dev),
                                _f32(self.norm_f2.bias, dev), self.norm_f2.eps),
                         "f3": (_f32(self.f3_weight, dev).reshape(1), _f32(self.norm_f3.weight, dev),
                                _f32(self.norm_f3.bias, dev), self.norm_f3.eps)}
        else:
            # stem: skip conv and first bottleneck conv of block1 concatenated, fp32
            bt0 = pk["b1"]["bott"][0]
            wskip = pk["b1"]["skip"]["conv"].weight.detach().to(dev).flatten(1).float()
            wmid = bt0["conv0"].weight.detach().to(dev).flatten(1).float()
            pk["stem"] = {"w": torch.cat([wskip, wmid], 0).contiguous(),
                          "s": torch.cat([pk["b1"]["skip"]["s"], bt0["s1"]]).contiguous(),
                          "b": torch.cat([pk["b1"]["skip"]["b"], bt0["b1"]]).contiguous(),
                          "n_skip": wskip.shape[0], "n_mid": wmid.shape[0]}
        for name in (("b1", "b2", "b3") if self.use_backbone else ("b2", "b3")):
            if name not in pk:
                continue
            blk = pk[name]
            for bt in blk["bott"]:
                bt["w0"] = _conv_w_bf16(bt["conv0"], dev)
            if "skip" in blk:
                blk["skip"]["w"] = _conv_w_bf16(blk["skip"]["conv"], dev)
                b0 = blk["bott"][0]
                # Tail conv with the residual folded into the contraction: out = [s*W7 | I] . [t ; skip] + b, i.e. the
                # identity branch enters as extra K channels with exact unit weights (fp32 accumulation, so the sum is
                # what an fp32 residual add gives).  The epilogue then has no residual to fetch and the 256-wide tile
                # becomes available.  Used while the widened contraction stays short (mid + Cout <= 512: block2,
                # 0.32 ms instead of 0.39 per launch at B = 1024); block3's 768-long contraction would make its tail
                # tensor bound (0.91 ms against 0.84 with the residual in the epilogue), so it keeps the epilogue form.
                last = blk["bott"][-1]
                w7 = last["conv7_f32"] * last["s8"][:, None]
                co = w7.shape[0]
                blk["tail_cat"] = {"w": torch.cat([w7, torch.eye(co, device=dev)], 1).to(torch.bfloat16).contiguous(),
                                   "b": last["b8"], "mid": w7.shape[1]}
                blk["fused_in"] = {"w": torch.cat([blk["skip"]["w"], b0["w0"]], 0).contiguous(),
                                   "s": torch.cat([blk["skip"]["s"], b0["s1"]]).contiguous(),
                                   "b": torch.cat([blk["skip"]["b"], b0["b1"]]).contiguous(),
                                   "n_split": blk["skip"]["w"].shape[0]}
        if not self.use_backbone:
            for bt in pk["b1"]["bott"][1:]:
                bt["w0"] = _conv_w_bf16(bt["conv0"], dev)
        if self.modality_attention is not None:
            pk["mod_se"] = _se_pack(self.modality_attention, dev)
        if self.mask_enabled:
            # the aligner feeding the mask head: f1 -> f2 for mask_stage f2, f2 -> f3 for f3, none for f1
            al = {"f1": nn.Identity(), "f2": self.f1_to_f2.proj, "f3": self.f2_to_f3.proj}[self.mask_stage]
            if isinstance(al, nn.Identity):  # equal channel counts (the ViT path) or mask_stage f1
                aw = s = b = None
            else:
                aw = _conv_w_bf16(al[0], dev)
                s, b = _bn_fold(al[1], dev)
            mh, ma = self.mask_head, self.mask_spatial_attention
            mproc = ma.mask_processor
            pk["mask"] = {
                "align_w": aw, "align_s": s, "align_b": b,
                "pre_w": _conv_w_bf16(mh.pre, dev), "pre_b": _f32(mh.pre.bias, dev),
                "down": _mask_down_pack(mh, dev),
                "out_w": _f32(mh.out.weight.flatten(), dev), "out_b": _f32(mh.out.bias, dev),
                "out_b_host": float(mh.out.bias.detach().float().cpu().item()),
                "attn": (mproc[0].out_channels, _f32(mproc[0].weight.flatten(), dev), _f32(mproc[1].weight, dev),
                         _f32(mproc[1].bias, dev), _f32(mproc[3].weight.flatten(), dev), _f32(mproc[3].bias, dev),
                         mproc[1].eps),
                "gamma": _f32(ma.gamma, dev).reshape(1),
            }
        pk["head"] = {"w": _f32(self.classification_head.fc.weight, dev), "b": _f32(self.classification_head.fc.bias, dev)}
        pk["proj"] = {n: _proj_pack(getattr(self, n), dev) for n in ("proj_f1", "proj_f2", "proj_r1", "proj_r2")}
        self._pack_cache = (sig, pk)
        return pk

    # ---------------------------------------------------------------- forward ----
    def _run_block(self, pk, mid, skip, need_recon, cat=None):
        """`mid` = output of the first bottleneck conv (+BN+GELU); `skip` = identity branch (both NHWC bf16), or
        `cat` = the tail GEMM's K-concatenated input whose upper channels already hold the identity branch."""
        botts = pk["bott"]
        dev = mid.device
        t = mid
        for i, bt in enumerate(botts):  # repeat_blocks bottlenecks in sequence (reference :298-310)
            if i > 0:  # later repeats start from the previous repeat's (un-activated) output
                st = pk.get("stride", 1) if pk.get("downsample_each_repeat", False) else 1
                t = nat.conv_gemm(t, bt["w0"], taps=1, scale=bt["s1"], bias=bt["b1"], act=1, stride=st,
                                  dropout=self._drop(1) if self._drop else None)
            last_into_cat = cat is not None and i + 1 == len(botts)
            t = nat.conv_gemm(t, bt["w4"], taps=9, scale=bt["s5"], bias=bt["b5"], act=1,
                              out=cat[..., :pk["tail_cat"]["mid"]] if last_into_cat else None)
            if i + 1 < len(botts):
                t = nat.conv_gemm(t, bt["w7"], taps=1, scale=bt["s8"], bias=bt["b8"], act=0)
        bt = botts[-1]
        B, H, W, _ = t.shape
        cout = bt["w7"].shape[0]
        drop = self._drop(1) if self._drop else None  # Dropout after GELU(out + identity), before SE (:305-306)
        if cat is not None:
            out, gap = _conv_gap(cat, pk["tail_cat"]["w"], taps=1, bias=pk["tail_cat"]["b"], act=1, dropout=drop)
        else:
            out, gap = _conv_gap(t, bt["w7"], taps=1, scale=bt["s8"], bias=bt["b8"], res=skip, res_mode=1, act=1,
                                 dropout=drop)
        gate = None
        if "se" in pk:
            se = pk["se"]
            gate = torch.empty((B, cout), dtype=torch.float32, device=dev)
            nat.se_gate(gap, H * W, se["w1t"], se["b1"], se["w2t"], se["b2"], gate)
            nat.scale_map(out, out, gate=gate)
        rec = _recon(pk["recon"], out) if (need_recon and "recon" in pk) else None
        return out, rec, gap, gate

    def _block_from_map(self, pk, x, need_recon):
        bt = pk["bott"][0]
        if "skip" in pk:
            # skip conv and first bottleneck conv read the same map: one GEMM, two output segments
            f = pk["fused_in"]
            st = pk.get("stride", 1)
            if "tail_cat" in pk and pk["tail_cat"]["w"].shape[1] <= 512:
                # the skip segment lands in the upper channels of the tail GEMM's K-concatenated input
                tc = pk["tail_cat"]
                B, H, W, _ = x.shape
                cat = torch.empty((B, H // st, W // st, tc["mid"] + f["n_split"]), dtype=torch.bfloat16, device=x.device)
                _, mid = nat.conv_gemm(x, f["w"], taps=1, scale=f["s"], bias=f["b"], act=0, n_split=f["n_split"],
                                       act2=1, stride=st, out=cat[..., tc["mid"]:],
                                       dropout=self._drop(2) if self._drop else None)
                return self._run_block(pk, mid, None, need_recon, cat=cat)
            skip, mid = nat.conv_gemm(x, f["w"], taps=1, scale=f["s"], bias=f["b"], act=0, n_split=f["n_split"],
                                      act2=1, stride=st, dropout=self._drop(2) if self._drop else None)
        else:
            skip = x
            mid = nat.conv_gemm(x, bt["w0"], taps=1, scale=bt["s1"], bias=bt["b1"], act=1,
                                dropout=self._drop(1) if self._drop else None)
        return self._run_block(pk, mid, skip, need_recon)

    def _mask_stage(self, mk, feat, prev):
        """Mask head on `feat` (+ the aligned previous-stage map, reference :682-684 / :696-698) and the mask-guided
        modulation feat *= 1 + gamma * A in place (:75-97).  Returns (mask_pred [B,1,S,S], attention map)."""
        B, Hm, Wm, _ = feat.shape
        dev = feat.device
        if prev is None:
            m_in = feat
        elif mk["align_w"] is None:
            m_in = nat.add_maps(feat, prev)
        else:
            m_in = nat.conv_gemm(prev, mk["align_w"], taps=1, scale=mk["align_s"], bias=mk["align_b"], act=1,
                                 res=feat, res_mode=2)
        mask_pred = _mask_head(mk, m_in, self.mask_size)
        mask_at_map = mask_pred
        if mask_pred.shape[-1] != Wm or mask_pred.shape[-2] != Hm:
            # MaskGuidedSpatialAttention resizes the prediction to the feature grid (:80-88)
            mask_at_map = torch.empty((B, 1, Hm, Wm), dtype=torch.float32, device=dev)
            nat.resize_bilinear_c1(mask_pred.view(B, *mask_pred.shape[-2:]), mask_at_map.view(B, Hm, Wm))
        attn_map = torch.empty((B, 1, Hm, Wm), dtype=torch.float32, device=dev)
        nat.mask_attention(mask_at_map, mk["attn"], attn_map)
        nat.scale_map(feat, feat, attn=attn_map, gamma=mk["gamma"])
        return mask_pred, attn_map

    def _project(self, pp, src, up2):
        if "w0_vec" in pp:  # 1-channel fp32 source map
            B, H, W = src.shape
            g = torch.empty((B, H, W, pp["w0_vec"].numel()), dtype=torch.bfloat16, device=src.device)
            nat.lift_c1(src, pp["w0_vec"], pp["s0"], pp["b0"], g)
        else:
            g = nat.conv_gemm(src, pp["w0"], taps=1, scale=pp["s0"], bias=pp["b0"], act=1)
        return nat.conv_gemm(g, pp["w3"], taps=1, scale=pp["s3"], bias=pp["b3"], act=1, up2=up2)

    def _project_pooled(self, pp, src):
        """proj(AdaptiveAvgPool2d(proj_dim)(src)) for any map size (reference :707-715).  The pool is an average
        and the projector's first 1x1 conv + BatchNorm is affine per pixel, so they commute: the conv runs on
        the small map, the pool (fused with the GELU) writes proj_dim^2 x 64 channels instead of
        proj_dim^2 x C, and the second 1x1 layer runs at the pooled size."""
        pd = self.proj_dim
        if "w0_vec" in pp:
            r = nat.adaptive_pool(src, pd)                      # [B,pd,pd] fp32
            g = torch.empty((*r.shape, pp["w0_vec"].numel()), dtype=torch.bfloat16, device=src.device)
            nat.lift_c1(r, pp["w0_vec"], pp["s0"], pp["b0"], g)
        else:
            y = nat.conv_gemm(src, pp["w0"], taps=1, scale=pp["s0"], bias=pp["b0"], act=0)
            g = nat.adaptive_pool(y, pd, act=1)
        return nat.conv_gemm(g, pp["w3"], taps=1, scale=pp["s3"], bias=pp["b3"], act=1)

    def _backbone_features(self, pk, x, plane_mean):
        """Modality attention + BackboneAdapter (reference :645-657, :401-476): returns (f1_b, f2_b, f3_b, gate)."""
        B, C, H, W = x.shape
        dev = x.device
        gate = None
        if "mod_se" in pk:
            if plane_mean is None:
                plane_mean = torch.empty(B * C, dtype=torch.float32, device=dev)
                nat.plane_mean(x, B * C, H * W, plane_mean)
            ms = pk["mod_se"]
            gate = torch.empty((B, C), dtype=torch.float32, device=dev)
            nat.se_gate(plane_mean.view(B, C), 1, ms["w1t"], ms["b1"], ms["w2t"], ms["b2"], gate)
        cats = self.backbone.forward_chains(x, self.selected_indices_chains, gate)
        outs = []
        for nk, cat in zip(pk["necks"], cats):
            t = nat.conv_gemm(cat, nk["w0"], taps=9, scale=nk["s0"], bias=nk["b0"], act=1)
            outs.append(nat.conv_gemm(t, nk["w3"], taps=9, scale=nk["s3"], bias=nk["b3"], act=1))
        return outs[0], outs[1], outs[2], gate

    # The reference wraps its models in torch.compile(backend='inductor') when parameters['compile'] is set
    # (code/run_training.py:90-91, :242-244).  The forward below is a schedule of C-ABI launches, nothing Dynamo could
    # trace: it is marked opaque, so a compiled wrapper of the module runs exactly this code (no graph breaks to
    # discover, no recompilations).
    @torch.compiler.disable
    def forward(self, x, masks=None, plane_mean=None, input_norm=None):
        """x [B,C,H,W] normalised fp32.  `plane_mean` (optional, [B*C] fp32) is the per-plane mean the
        normaliser kernels can emit, which saves one pass over x.  `input_norm` (with plane_mean): x is the RAW
        input and the normalisation runs inside the first layer's operand load (DWINormalize.fused_params /
        DCENormalize.fused_params; eval mode, CNN encoders)."""
        if not x.is_cuda:
            raise nat.B200NativeError("ModelMaskHeadBackbone.forward needs a CUDA tensor (no CPU path)")
        if self.training:
            # train mode (reference :298-316, :645-733 under nn.Module.train()): batch-statistic BatchNorm with
            # running-statistics update, active dropout, and a torch-autograd node whose backward runs the explicit
            # backward pass of train_graph on the training kernels
            from train_graph import encoder_train_forward_autograd

            return encoder_train_forward_autograd(self, x)
        p_drop = self._mc_dropout_p()
        dev = x.device
        pk = self._packed(dev)
        self._drop = None
        if p_drop > 0 or (self.use_hybrid_transformer and _transformer_dropouts(pk["tr"])):
            # per-launch seeds: (model seed, forward count, launch count)
            self._mc_calls += 1
            base = (self._mc_seed * 0x9E3779B97F4A7C15 + self._mc_calls * 0xD1B54A32D192ED03) & 0xFFFFFFFFFFFFFFFF
            counter = [0]

            def _drop(segments=1, p=p_drop):
                """(p, seed, segments) of the next dropout launch, or None when p is 0 (p defaults to the CNN blocks')."""
                if p <= 0:
                    return None
                counter[0] += 1
                return (p, (base + counter[0] * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF, segments)

            self._drop = _drop
        full = self.aux_mode == "full"
        x = x.contiguous().float()
        B, C, H, W = x.shape
        mod_attn = None
        f2_b = f3_b = None
        if input_norm is not None and (self.use_backbone or "mod_se" not in pk):
            raise NotImplementedError("input_norm: the fused first layer is the CNN encoders' stem (modality attention on)")
        if self.use_backbone:
            f1_b, f2_b, f3_b, mod_attn = self._backbone_features(pk, x, plane_mean)
            f1, r1, _, _ = self._block_from_map(pk["b1"], f1_b, full)
            Ho, Wo = f1.shape[1], f1.shape[2]
        else:
            st = pk["stem"]
            stride = self.block1.stride
            Ho, Wo = H // stride, W // stride
            se = None
            if "mod_se" in pk:
                if plane_mean is None:
                    plane_mean = torch.empty(B * C, dtype=torch.float32, device=dev)
                    nat.plane_mean(x, B * C, H * W, plane_mean)
                ms = pk["mod_se"]
                se = (ms["w1"], ms["b1"], ms["w2"], ms["b2"])
                mod_attn = torch.empty((B, C), dtype=torch.float32, device=dev)
            skip1 = torch.empty((B, Ho, Wo, st["n_skip"]), dtype=torch.bfloat16, device=dev)
            mid1 = torch.empty((B, Ho, Wo, st["n_mid"]), dtype=torch.bfloat16, device=dev)
            if input_norm is not None and plane_mean is None:
                raise ValueError("input_norm needs the plane means of the normalised values (fused_params returns both)")
            nat.stem(x, stride, plane_mean, se, st["w"], st["s"], st["b"], st["n_skip"], st["n_mid"], skip1, mid1,
                     mod_attn, dropout=self._drop(1)[:2] if self._drop and p_drop > 0 else None, input_norm=input_norm)
            f1, r1, _, _ = self._run_block(pk["b1"], mid1, skip1, full)

        mask_pred = attn_map = None
        if self.mask_enabled and self.mask_stage == "f1":                       # reference :668-670
            mask_pred, attn_map = self._mask_stage(pk["mask"], f1, None)
        f2_in = f1
        if self.use_backbone:  # reference :673-675
            f2_in = nat.mix_instnorm(f2_b, f1, *pk["mix"]["f2"])
        f2, r2, _, _ = self._block_from_map(pk["b2"], f2_in, full)
        if self.mask_enabled and self.mask_stage == "f2":                       # reference :681-685
            mask_pred, attn_map = self._mask_stage(pk["mask"], f2, f1)
        if self.use_hybrid_transformer:
            f3, gap3 = _transformer_stage(pk["tr"], f2, self._drop)  # reference :702-703
            gate3 = None
        else:
            f3_in = f2
            if self.use_backbone:  # reference :688-690
                f3_in = nat.mix_instnorm(f3_b, f2, *pk["mix"]["f3"])
            f3, _, gap3, gate3 = self._block_from_map(pk["b3"], f3_in, False)
            if self.mask_enabled and self.mask_stage == "f3":                   # reference :695-699
                mask_pred, attn_map = self._mask_stage(pk["mask"], f3, f2)
                gap3, gate3 = nat.channel_sums(f3), None  # the classifier pools the modulated map
        npix3 = f3.shape[1] * f3.shape[2]

        logits = None
        p1 = p1r = p2 = p2r = None
        if full:
            logits = torch.empty((B, self.num_classes), dtype=torch.float32, device=dev)
            nat.cls_head(gap3, gate3, npix3, pk["head"]["w"], pk["head"]["b"], self.classification_head.normalize,
                         logits)
            pj = pk["proj"]

            def proj(pp, src):
                hs, ws = src.shape[1], src.shape[2]
                if self.proj_dim in (hs, 2 * hs) and hs == ws and _staged_tiles(hs, ws):
                    # AdaptiveAvgPool2d to the same size is the identity, to 2x the size a 2x2 replication
                    return self._project(pp, src, self.proj_dim == 2 * hs)
                return self._project_pooled(pp, src)

            p1 = _nchw(proj(pj["proj_f1"], f1))
            p2 = _nchw(proj(pj["proj_f2"], f2))
            p1r = _nchw(proj(pj["proj_r1"], r1))
            p2r = _nchw(proj(pj["proj_r2"], r2))
        aux = {
            "raw_feats": [_nchw(f1), _nchw(f2), _nchw(f3)],
            "recon_feats": [r1.unsqueeze(1) if r1 is not None else None, r2.unsqueeze(1) if r2 is not None else None],
            "proj_pairs": [p1, p1r, p2, p2r],
            "mask_attn_map": attn_map,
            "mod_attn_map": mod_attn.view(B, C, 1, 1) if mod_attn is not None else None,
        }
        return logits, aux, mask_pred


# --------------------------------------------------------------------------------------
# fusion
# --------------------------------------------------------------------------------------
def _bilinear_axis_weights(n_in, n_out):
    """Mean weight each source cell receives under F.interpolate(bilinear, align_corners=False)."""
    w = [0.0] * n_in
    scale = n_in / n_out
    for d in range(n_out):
        s = max((d + 0.5) * scale - 0.5, 0.0)
        i0 = int(s)
        i1 = min(i0 + 1, n_in - 1)
        lam = s - i0
        w[i0] += (1.0 - lam) / n_out
        w[i1] += lam / n_out
    return w


class FusionModel(_PackedWeightsMixin, nn.Module):
    """Late-fusion head (reference :821-1000).  The reference's cat -> fusion_conv_reduce -> refine
    branch (:935-940) never reaches an output, so it is not evaluated (its parameters exist for
    state_dict compatibility)."""

    def __init__(self, parameters_dict):
        super().__init__()
        fc = parameters_dict["fusion_model_parameters"]
        fs = fc["fusion_specific_parameters"]
        self.dim = parameters_dict["dim"]
        _only_2d(self.dim)
        self.num_classes = parameters_dict["class_num"]
        self.fusion_channels = fs["fusion_channels"]
        self.token_pool = fs["token_pool"]
        self.mha_heads = fs["mha_heads"]
        self.dwi_ch, self.dce_ch = fs["dwi_out_channels"], fs["dce_out_channels"]
        self.use_cross_attention = fs["use_cross_attention"]
        self.use_mask_attention = fs["use_mask_attention"]
        self.fusion_recon_ch = fs["fusion_recon_ch"]
        self.proj_dim = fc["proj_dim"]
        self.mask_size = fc["mask_parameters"]["mask_target_size"][0]
        self.dropout = fc["dropout"]
        self.use_se_in_fusion = fc["use_se"]
        self.aux_mode = "full"
        c = self.fusion_channels
        self.proj_in_dwi = nn.Conv2d(self.dwi_ch, c, 1, bias=False) if self.dwi_ch != c else nn.Identity()
        self.proj_in_dce = nn.Conv2d(self.dce_ch, c, 1, bias=False) if self.dce_ch != c else nn.Identity()
        self.fusion_conv_reduce = FusionReduce(2 * c, c, dim=self.dim)
        self.refine_act = nn.GELU()
        self.fusion_se = SEBlock(c, reduction=2, dim=self.dim) if self.use_se_in_fusion else None
        self.gating = GatingAttention(feat_dim=c, use_mask_attention=self.use_mask_attention, dim=self.dim)
        self.refine = ResNetLiteBlock_withRecon(in_ch=c, out_ch=c, dim=self.dim, dropout=self.dropout, mid_squeeze=2)
        if self.use_cross_attention:
            self.cross_attn_block = CrossAttentionBlock(c, num_heads=self.mha_heads)
        self.mask_head = MaskHeadResize(in_ch=c, out_size=self.mask_size, dim=self.dim)
        self.fusion_reconstruct = ReconHead(in_ch=c, recon_ch=self.fusion_recon_ch, upsample=False, dim=self.dim)
        self.classifier = nn.Sequential(nn.AdaptiveAvgPool2d((1, 1)), nn.Flatten(), nn.Linear(c, self.num_classes))
        self.projF = Projector(in_ch=c, proj_dim=self.proj_dim, dim=self.dim)
        self._pack_cache = None

    def _packed(self, dev, H, W):
        sig = (str(dev), H, W, _state_signature(self))
        if self._pack_cache is not None and self._pack_cache[0] == sig:
            return self._pack_cache[1]
        if isinstance(self.proj_in_dwi, nn.Identity) or isinstance(self.proj_in_dce, nn.Identity):
            raise NotImplementedError("encoder channels == fusion_channels (identity proj_in) is not built")
        c = self.fusion_channels
        hp, wp = self.token_pool
        keep = {}
        w = nat.FusionWeights()
        w.C, w.T, w.heads, w.num_classes = c, hp * wp, self.mha_heads, self.num_classes
        w.use_cross_attention = int(self.use_cross_attention)
        w.use_mask_attention = int(self.use_mask_attention)
        w.use_se = int(self.fusion_se is not None)

        def put(name, t):
            keep[name] = _f32(t, dev)
            setattr(w, name, keep[name].data_ptr())

        put("gate_w", self.gating.fc.weight)
        put("gate_b", self.gating.fc.bias)
        if self.use_cross_attention:
            ca = self.cross_attn_block
            put("in_proj_wt", ca.cross_attn.in_proj_weight.t())
            put("in_proj_b", ca.cross_attn.in_proj_bias)
            put("out_proj_wt", ca.cross_attn.out_proj.weight.t())
            put("out_proj_b", ca.cross_attn.out_proj.bias)
            put("ln_w", ca.attn_ffn[0].weight)
            put("ln_b", ca.attn_ffn[0].bias)
            w.ln_eps = ca.attn_ffn[0].eps
            put("ffn1_wt", ca.attn_ffn[1].weight.t())
            put("ffn1_b", ca.attn_ffn[1].bias)
            put("ffn2_wt", ca.attn_ffn[3].weight.t())
            put("ffn2_b", ca.attn_ffn[3].bias)
            ah, aw = _bilinear_axis_weights(hp, H), _bilinear_axis_weights(wp, W)
            put("up_coef", torch.tensor([ah[i] * aw[j] for i in range(hp) for j in range(wp)]))
        if self.fusion_se is not None:
            se = _se_pack(self.fusion_se, dev)
            w.se_mid = se["b1"].numel()
            put("se_w1t", se["w1t"])
            put("se_b1", se["b1"])
            put("se_w2t", se["w2t"])
            put("se_b2", se["b2"])
        put("cls_w", self.classifier[2].weight)
        put("cls_b", self.classifier[2].bias)
        mh = self.mask_head
        pk = {"w": w, "keep": keep,
              "in_dwi": _conv_w_bf16(self.proj_in_dwi, dev), "in_dce": _conv_w_bf16(self.proj_in_dce, dev),
              "mask": {"pre_w": _conv_w_bf16(mh.pre, dev), "pre_b": _f32(mh.pre.bias, dev),
                       "down": _mask_down_pack(mh, dev), "out_w": _f32(mh.out.weight.flatten(), dev),
                       "out_b_host": float(mh.out.bias.detach().float().cpu().item())},
              "recon": _recon_pack(self.fusion_reconstruct, dev), "projF": _proj_pack(self.projF, dev)}
        self._pack_cache = (sig, pk)
        return pk

    @torch.compiler.disable  # see ModelMaskHeadBackbone.forward
    def forward(self, raw_feats_dwi, raw_feats_dce, dwi_mask_pred=None, dce_mask_pred=None):
        if self.training:
            if not raw_feats_dwi[-1].is_cuda:
                raise nat.B200NativeError("feature maps must be CUDA tensors (no CPU path)")
            from train_graph import fusion_train_forward_autograd

            return fusion_train_forward_autograd(self, raw_feats_dwi, raw_feats_dce, dwi_mask_pred, dce_mask_pred)
        f3d, f3c = _as_nhwc_bf16(raw_feats_dwi[-1]), _as_nhwc_bf16(raw_feats_dce[-1])
        B, H, W, _ = f3d.shape
        dev = f3d.device
        pk = self._packed(dev, H, W)
        c = self.fusion_channels
        hp, wp = self.token_pool
        full = self.aux_mode == "full"
        if self.use_mask_attention and (dwi_mask_pred is None or dce_mask_pred is None):
            # the reference feeds a 2C vector into a (2C+2)-input Linear in this case and raises too
            raise RuntimeError("use_mask_attention needs both encoder mask predictions")
        p_dwi, pv_d = _conv_gap(f3d, pk["in_dwi"], taps=1)
        p_dce, pv_c = _conv_gap(f3c, pk["in_dce"], taps=1)
        tok_d = tok_c = attn_w = lowres = None
        if self.use_cross_attention:
            tok_d = torch.empty((B, hp * wp, c), dtype=torch.float32, device=dev)
            tok_c = torch.empty_like(tok_d)
            nat.fusion_tokens(p_dwi, hp, wp, tok_d)
            nat.fusion_tokens(p_dce, hp, wp, tok_c)
            attn_w = torch.empty((B, hp * wp, hp * wp), dtype=torch.float32, device=dev)
            lowres = torch.empty((B, hp * wp, c), dtype=torch.float32, device=dev)
        gating = torch.empty((B, 2), dtype=torch.float32, device=dev)
        gate = torch.empty((B, c), dtype=torch.float32, device=dev)
        logits = torch.empty((B, self.num_classes), dtype=torch.float32, device=dev)
        md = mc = None
        npix_mask = 0
        if self.use_mask_attention:
            md = dwi_mask_pred.contiguous().float()
            mc = dce_mask_pred.contiguous().float()
            npix_mask = md[0].numel()
        nat.fusion_core(pk["w"], B, pv_d, pv_c, H * W, md, mc, npix_mask, tok_d, tok_c, gating, attn_w, lowres, gate,
                        logits)
        mask_logits = recon = proj = None
        if full:  # (the logits come from the pooled vectors: the fused map only feeds the mask / recon / projector heads)
            fused = torch.empty((B, H, W, c), dtype=torch.bfloat16, device=dev)
            nat.fusion_mix(p_dwi, p_dce, gating, lowres, gate if self.fusion_se is not None else None, hp, wp, fused)
            mask_logits = _mask_head(pk["mask"], fused, self.mask_size)
            recon = _recon(pk["recon"], fused).unsqueeze(1)
            pj = pk["projF"]
            g = nat.conv_gemm(fused, pj["w0"], taps=1, scale=pj["s0"], bias=pj["b0"], act=1)
            proj = _nchw(nat.conv_gemm(g, pj["w3"], taps=1, scale=pj["s3"], bias=pj["b3"], act=1))
        aux = {"proj_fused": proj, "recon_fused": recon, "gating_weights": gating, "attn_weights": attn_w,
               "p_dwi": _nchw(p_dwi), "p_dce": _nchw(p_dce)}
        return logits, mask_logits, aux


# --------------------------------------------------------------------------------------
# initialisation (reference :1002-1023)
# --------------------------------------------------------------------------------------
def init_parameter(model):
    """Linear: Kaiming-uniform weight, zero bias.  BatchNorm: weight ~ N(1, 0.02), zero bias."""
    if isinstance(model, nn.Linear):
        if model.weight is not None:
            init.kaiming_uniform_(model.weight.data)
        if model.bias is not None:
            init.constant_(model.bias.data, 0)
    elif isinstance(model, (nn.BatchNorm1d, nn.BatchNorm2d, nn.BatchNorm3d)):
        if model.weight is not None:
            init.normal_(model.weight.data, mean=1, std=0.02)
        if model.bias is not None:
            init.constant_(model.bias.data, 0)


def initialize_model(model, requires_grad):
    for param in model.parameters():
        param.requires_grad = requires_grad
    model.apply(init_parameter)
    for mod in model.modules():  # init_parameter writes through .data: the packed copies are stale now
        if isinstance(mod, _PackedWeightsMixin):
            mod.invalidate_packed()
    return model
