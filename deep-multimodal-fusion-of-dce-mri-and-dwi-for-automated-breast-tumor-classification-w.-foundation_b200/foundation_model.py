"""B200-native drop-in for the reference's ``foundation_model``: the ViT-B/16 and ResNet-50 backbone branches.

``build_medical_backbone(parameters, device, method, in_channels)`` keeps the reference contract
(/root/reference/code/foundation_model.py:490-577): it returns an ``nn.Module`` with
``.feature_info.channels()/.reduction()``, ``.output_dims`` and ``forward(x) -> list[NCHW maps]`` and
mutates ``parameters[f"{method}_model_parameters"]`` the way the reference's branches do - ViT (:526-545):
``backbone_index_lists=[[0,1,2],[3,4,5,6],[7,8,9,10,11]]``, ``downsample=(False,)*3``, ``channels=(768,)*3``,
``transformer_backbone=True``; resnet50 / radimagenet (:503-524, :547-569): ``backbone_index_lists=[[0],[1],[2,3]]``,
``downsample=(True, False, False)``, ``downsample_each_repeat=False``.

The reference gets the networks from timm (``timm.create_model("vit_base_patch16_224", features_only=True,
out_indices=0..11, ...)`` :371-431; ``timm.create_model("resnet50", features_only=True, output_stride=8,
out_indices=(1,2,3,4), ...)`` :15-68, :243-250).  timm is an un-vendored, un-pinned dependency that is absent
here, so this module carries its own feature extractors with timm's parameter names - a timm (or, re-keyed,
RadImageNet) checkpoint's ``state_dict`` loads unchanged - and runs them on the sm_100a kernels:

* ``B200ViTBackbone``: patchify + one GEMM for the patch embedding, an fp32 residual stream, LayerNorm (eps 1e-6),
  per-head Q.K^T with the softmax numerator fused into the GEMM epilogue (197 keys masked inside a 256-wide tile),
  P.V with the 1/rowsum applied to the fp32 accumulator, MLP with a fused GELU.
* ``B200ResNetBackbone``: the 7x7 stem as shared-memory im2col + one GEMM, max-pool, then the 16 bottlenecks as
  implicit GEMMs with folded BatchNorm, ReLU, stride / dilation and the residual in the epilogue.

Parity for the backbones themselves is UNPINNED (no timm to compare with); the oracles are restatements
cross-checked against torchvision's VisionTransformer / ResNet (oracle/backbone_oracle.py).  ResNet-50d,
ResNet-101 and UNI2-h are not built.  No pretrained weights can be fetched offline: parameters are randomly
initialised unless a state dict (or a local ``pretrained_path``) is loaded.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

import b200_native as nat

__all__ = ["build_medical_backbone", "build_vit_dino_backbone", "build_radimagenet_backbone", "build_imagenet_backbone",
           "B200ViTBackbone", "B200ResNetBackbone"]

VIT_NAMES = ("vit_base_patch16_224", "dino_vitbase16_pretrain", "dino_vitbase16_pretrained")
RESNET_NAMES = ("resnet50", "radimagenet", "radimagenet_resnet50")


class _FeatureInfo:
    def __init__(self, channels, reductions):
        self._c, self._r = list(channels), list(reductions)

    def channels(self):
        return list(self._c)

    def reduction(self):
        return list(self._r)


class _PatchEmbed(nn.Module):
    def __init__(self, in_chans, embed, patch):
        super().__init__()
        self.proj = nn.Conv2d(in_chans, embed, kernel_size=patch, stride=patch)


class _Attention(nn.Module):
    def __init__(self, embed, heads):
        super().__init__()
        self.num_heads = heads
        self.qkv = nn.Linear(embed, 3 * embed, bias=True)
        self.proj = nn.Linear(embed, embed)


class _Mlp(nn.Module):
    def __init__(self, embed, hidden):
        super().__init__()
        self.fc1 = nn.Linear(embed, hidden)
        self.fc2 = nn.Linear(hidden, embed)


class _Block(nn.Module):
    def __init__(self, embed, heads, hidden):
        super().__init__()
        self.norm1 = nn.LayerNorm(embed, eps=1e-6)
        self.attn = _Attention(embed, heads)
        self.norm2 = nn.LayerNorm(embed, eps=1e-6)
        self.mlp = _Mlp(embed, hidden)


def _f32(t, dev):
    return t.detach().to(device=dev, dtype=torch.float32).contiguous()


def _bf16(t, dev):
    return t.detach().to(device=dev, dtype=torch.bfloat16).contiguous()


class B200ViTBackbone(nn.Module):
    """ViT-B/16 `features_only` backbone: forward(x[B,C,H,W]) -> 12 maps [B,768,H/16,W/16] (bf16,
    channels_last views), cls token stripped, no final norm - what timm's FeatureGetterNet returns."""

    def __init__(self, in_chans=3, img_size=224, patch_size=16, embed_dim=768, depth=12, num_heads=12, mlp_ratio=4.0,
                 out_indices=None):
        super().__init__()
        self.patch_size, self.embed_dim, self.img_size = patch_size, embed_dim, img_size
        self.grid = img_size // patch_size
        self.out_indices = list(range(depth)) if out_indices is None else list(out_indices)
        self.patch_embed = _PatchEmbed(in_chans, embed_dim, patch_size)
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.pos_embed = nn.Parameter(torch.randn(1, self.grid * self.grid + 1, embed_dim) * 0.02)
        self.blocks = nn.ModuleList([_Block(embed_dim, num_heads, int(embed_dim * mlp_ratio)) for _ in range(depth)])
        self.norm = nn.LayerNorm(embed_dim, eps=1e-6)  # present in timm's model; not applied to features
        self.feature_info = _FeatureInfo([embed_dim] * len(self.out_indices), [patch_size] * len(self.out_indices))
        self.output_dims = [embed_dim] * len(self.out_indices)
        self._pack_cache = None

    def _packed(self, dev):
        sig = (str(dev), tuple((t.data_ptr(), t._version) for t in self.parameters()))
        if self._pack_cache is not None and self._pack_cache[0] == sig:
            return self._pack_cache[1]
        E = self.embed_dim
        pk = {"pe_w": _bf16(self.patch_embed.proj.weight.flatten(1), dev), "pe_b": _f32(self.patch_embed.proj.bias, dev),
              "cls": _f32(self.cls_token.flatten(), dev), "pos": _f32(self.pos_embed[0], dev), "layers": []}
        for blk in self.blocks:
            wqkv, bqkv = blk.attn.qkv.weight, blk.attn.qkv.bias
            pk["layers"].append({
                "heads": blk.attn.num_heads, "dh": E // blk.attn.num_heads,
                "ln1": (_f32(blk.norm1.weight, dev), _f32(blk.norm1.bias, dev), blk.norm1.eps),
                "ln2": (_f32(blk.norm2.weight, dev), _f32(blk.norm2.bias, dev), blk.norm2.eps),
                "wqkv": _bf16(wqkv, dev), "bqkv": _f32(bqkv, dev),
                "wproj": _bf16(blk.attn.proj.weight, dev), "bproj": _f32(blk.attn.proj.bias, dev),
                "wfc1": _bf16(blk.mlp.fc1.weight, dev), "bfc1": _f32(blk.mlp.fc1.bias, dev),
                "wfc2": _bf16(blk.mlp.fc2.weight, dev), "bfc2": _f32(blk.mlp.fc2.bias, dev)})
        self._pack_cache = (sig, pk)
        return pk

    @torch.no_grad()
    def forward(self, x):
        return self._run(x, None, None)

    @torch.no_grad()
    def forward_chains(self, x, chains, gate=None):
        """What BackboneAdapter needs (reference model_module.py:452-471): for every index chain the channel
        concatenation of its feature maps, as one NHWC bf16 buffer [B, g, g, len(chain)*E] that the blocks'
        outputs are written straight into (no torch.cat pass).  `gate` [B,C] fp32 is the modality-attention
        weight, applied while the image is cut into patches."""
        return self._run(x, gate, [list(c) for c in chains])

    def _run(self, x, gate, chains):
        if self.training:
            raise NotImplementedError("training-mode forward is not built in the B200 path yet; call .eval()")
        if not x.is_cuda:
            raise nat.B200NativeError("B200ViTBackbone.forward needs a CUDA tensor (no CPU path)")
        x = x.contiguous().float()
        B, C, H, W = x.shape
        P, E = self.patch_size, self.embed_dim
        if H != self.img_size or W != self.img_size:
            raise ValueError(f"expected {self.img_size}x{self.img_size} inputs (fixed position embedding)")
        g = self.grid
        n = g * g          # patch tokens
        N = n + 1          # + cls
        dev = x.device
        pk = self._packed(dev)
        K0 = C * P * P
        if K0 % 64 != 0:
            raise NotImplementedError("in_chans * patch^2 must be a multiple of 64")
        patches = torch.empty((B * n, K0), dtype=torch.bfloat16, device=dev)
        nat.patchify(x, P, patches, gate)
        emb = nat.linear(patches, pk["pe_w"], bias=pk["pe_b"])            # [B*n, E] bf16
        t = torch.empty((B * N, E), dtype=torch.float32, device=dev)      # fp32 residual stream
        nat.vit_tokens(emb, pk["cls"], pk["pos"], B, n, E, t)
        M = B * N
        h = torch.empty((M, E), dtype=torch.bfloat16, device=dev)
        qkv = torch.empty((M, 3 * E), dtype=torch.bfloat16, device=dev)
        o = torch.empty((M, E), dtype=torch.bfloat16, device=dev)
        u = torch.empty((M, pk["layers"][0]["wfc1"].shape[0]), dtype=torch.bfloat16, device=dev)
        heads, dh = pk["layers"][0]["heads"], pk["layers"][0]["dh"]
        feats = []
        bufs = None
        if chains is not None:
            bufs = [torch.empty((B, g, g, len(c) * E), dtype=torch.bfloat16, device=dev) for c in chains]
        for i, ly in enumerate(pk["layers"]):
            nat.layernorm(t, *ly["ln1"], out=h)
            nat.linear(h, ly["wqkv"], bias=ly["bqkv"], out=qkv)
            # softmax(q k^T / sqrt(d)) v per (case, head) in one launch: scores in TMEM, probabilities in shared memory
            nat.attention(qkv, o, B, N, heads, dh)
            t2 = nat.linear_f32(o, ly["wproj"], bias=ly["bproj"], res=t, res_mode=2, out_dtype=torch.float32)
            nat.layernorm(t2, *ly["ln2"], out=h)
            nat.linear(h, ly["wfc1"], bias=ly["bfc1"], act=1, out=u)
            t = nat.linear_f32(u, ly["wfc2"], bias=ly["bfc2"], res=t2, res_mode=2, out_dtype=torch.float32)
            if chains is not None:
                for ci, chain in enumerate(chains):
                    for slot, idx in enumerate(chain):
                        if self.out_indices[idx] == i:  # feats[idx] is block out_indices[idx]
                            nat.vit_feature(t, B, n, E, bufs[ci][..., slot * E:(slot + 1) * E], out_ld=len(chain) * E)
            elif i in self.out_indices:
                f = torch.empty((B, g, g, E), dtype=torch.bfloat16, device=dev)
                nat.vit_feature(t, B, n, E, f)
                feats.append(f.permute(0, 3, 1, 2))  # NCHW-shaped view of the NHWC buffer
        return feats if chains is None else bufs


# --------------------------------------------------------------------------------------
# ResNet-50 (timm / torchvision `resnet50`, v1.5: the stride sits on the 3x3 conv)
# --------------------------------------------------------------------------------------
class _Bottleneck(nn.Module):
    """keys conv1, bn1, conv2, bn2, conv3, bn3, downsample.{0,1} (timm / torchvision Bottleneck)."""

    def __init__(self, cin, planes, stride, dilation, downsample):
        super().__init__()
        self.conv1 = nn.Conv2d(cin, planes, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.conv2 = nn.Conv2d(planes, planes, 3, stride=stride, padding=dilation, dilation=dilation, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.conv3 = nn.Conv2d(planes, planes * 4, 1, bias=False)
        self.bn3 = nn.BatchNorm2d(planes * 4)
        self.downsample = None
        if downsample:
            self.downsample = nn.Sequential(nn.Conv2d(cin, planes * 4, 1, stride=stride, bias=False),
                                            nn.BatchNorm2d(planes * 4))
        self.stride, self.dilation = stride, dilation


def _bn_affine(bn, dev):
    g, b = _f32(bn.weight, dev), _f32(bn.bias, dev)
    m, v = _f32(bn.running_mean, dev), _f32(bn.running_var, dev)
    scale = g / torch.sqrt(v + bn.eps)
    return scale.contiguous(), (b - m * scale).contiguous()


def _conv_k_major(conv, dev):
    w = conv.weight.detach().to(dev)
    return w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).to(torch.bfloat16).contiguous()


class B200ResNetBackbone(nn.Module):
    """ResNet-50 `features_only` backbone as the reference builds it with timm (foundation_model.py:15-68, :220-312:
    `timm.create_model("resnet50", features_only=True, output_stride=8, out_indices=(1, 2, 3, 4), in_chans=C)`):
    forward(x[B,C,H,W]) -> [C2 (256, /4), C3 (512, /8), C4 (1024, /8, dilated), C5 (2048, /8, dilated)] as bf16
    channels_last views.  Parameter names are timm's / torchvision's (conv1, bn1, layerN.M.{conv1..bn3, downsample}),
    so resnet50 and (re-keyed, see map_rasool_to_timm_keys) RadImageNet checkpoints load unchanged.  Eval-mode only:
    BatchNorm is folded into the GEMM epilogues."""

    def __init__(self, in_chans=3, layers=(3, 4, 6, 3), output_stride=8, out_indices=(1, 2, 3, 4)):
        super().__init__()
        if output_stride not in (8, 16, 32):
            raise ValueError("output_stride must be 8, 16 or 32")
        self.conv1 = nn.Conv2d(in_chans, 64, 7, stride=2, padding=3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        self.out_indices = list(out_indices)
        if any(i not in (1, 2, 3, 4) for i in self.out_indices):
            raise NotImplementedError("only the C2..C5 features (out_indices 1..4) are built")
        cin, net_stride, dilation, prev_dilation = 64, 4, 1, 1
        reductions = []
        for li, (planes, n_blocks, stride) in enumerate(zip((64, 128, 256, 512), layers, (1, 2, 2, 2))):
            if net_stride >= output_stride:  # timm: trade the stride for dilation once the target stride is reached
                dilation *= stride
                stride = 1
            else:
                net_stride *= stride
            blocks = []
            for bi in range(n_blocks):
                blocks.append(_Bottleneck(cin, planes, stride if bi == 0 else 1, prev_dilation if bi == 0 else dilation,
                                          downsample=(bi == 0)))
                cin = planes * 4
            prev_dilation = dilation
            setattr(self, f"layer{li + 1}", nn.Sequential(*blocks))
            reductions.append(net_stride)
        chans = [256, 512, 1024, 2048]
        self.feature_info = _FeatureInfo([chans[i - 1] for i in self.out_indices], [reductions[i - 1] for i in self.out_indices])
        self.output_dims = self.feature_info.channels()
        self.expected_input, self.is_3d, self.foundation_model, self.transformer_backbone = "B, C, H, W", False, True, False
        self._pack_cache = None

    def _packed(self, dev):
        sig = (str(dev), tuple((t.data_ptr(), t._version) for t in list(self.parameters()) + list(self.buffers())))
        if self._pack_cache is not None and self._pack_cache[0] == sig:
            return self._pack_cache[1]
        s0, b0 = _bn_affine(self.bn1, dev)
        w = self.conv1.weight.detach().to(dev).float()
        kp = (w.shape[1] * 49 + 63) // 64 * 64   # conv1 as a GEMM over zero-padded im2col rows (Conv2d weight order)
        wg = torch.zeros((64, kp), dtype=torch.bfloat16, device=dev)
        wg[:, :w.shape[1] * 49] = w.flatten(1).to(torch.bfloat16)
        pk = {"stem": (s0, b0), "stem_gemm": (wg, kp), "layers": []}
        for li in range(4):
            blocks = []
            for blk in getattr(self, f"layer{li + 1}"):
                d = {"w1": _conv_k_major(blk.conv1, dev), "a1": _bn_affine(blk.bn1, dev),
                     "w2": _conv_k_major(blk.conv2, dev), "a2": _bn_affine(blk.bn2, dev),
                     "w3": _conv_k_major(blk.conv3, dev), "a3": _bn_affine(blk.bn3, dev),
                     "stride": blk.stride, "dilation": blk.dilation}
                if blk.downsample is not None:
                    d["wd"] = _conv_k_major(blk.downsample[0], dev)
                    d["ad"] = _bn_affine(blk.downsample[1], dev)
                blocks.append(d)
            pk["layers"].append(blocks)
        self._pack_cache = (sig, pk)
        return pk

    @torch.no_grad()
    def forward(self, x):
        return [f.permute(0, 3, 1, 2) for f in self._run(x, None, None)]

    @torch.no_grad()
    def forward_chains(self, x, chains, gate=None):
        """Per index chain the channel concatenation of its feature maps (BackboneAdapter, model_module.py:452-471),
        written in place: a layer's last bottleneck stores straight into its slice of the chain buffer."""
        return self._run(x, gate, [list(c) for c in chains])

    def _run(self, x, gate, chains):
        if self.training:
            raise NotImplementedError("training-mode forward is not built in the B200 path yet; call .eval()")
        if not x.is_cuda:
            raise nat.B200NativeError("B200ResNetBackbone.forward needs a CUDA tensor (no CPU path)")
        x = x.contiguous().float()
        dev = x.device
        pk = self._packed(dev)
        B = x.shape[0]
        # conv1 + bn1 + ReLU as one GEMM over the im2col rows (18.8 -> ~5 ms per 256-case step against the fp32 SIMT
        # direct convolution it replaced)
        wg, kp = pk["stem_gemm"]
        cols = nat.im2col7x7_s2(x, gate, kp)
        s0, b0 = pk["stem"]
        t = nat.linear(cols, wg, scale=s0, bias=b0, act=2).view(B, x.shape[2] // 2, x.shape[3] // 2, 64)
        t = nat.maxpool3x3_s2(t)   # [B, H/4, W/4, 64]
        chans = [256, 512, 1024, 2048]
        # where does feature fi (position in the returned list) have to land?
        dest = {}
        bufs = None
        if chains is not None:
            sizes = []
            for chain in chains:
                sizes.append(sum(self.feature_info.channels()[i] for i in chain))
            bufs = [None] * len(chains)
            for ci, chain in enumerate(chains):
                off = 0
                for fi in chain:
                    dest[fi] = (ci, off, sizes[ci])
                    off += self.feature_info.channels()[fi]
        feats = []
        for li, blocks in enumerate(pk["layers"]):
            fi = self.out_indices.index(li + 1) if (li + 1) in self.out_indices else None
            for bi, blk in enumerate(blocks):
                last = bi == len(blocks) - 1
                h = nat.conv_gemm(t, blk["w1"], taps=1, scale=blk["a1"][0], bias=blk["a1"][1], act=2)
                h = nat.conv_gemm(h, blk["w2"], taps=9, scale=blk["a2"][0], bias=blk["a2"][1], act=2,
                                  stride=blk["stride"], dilation=blk["dilation"])
                idn = t
                if "wd" in blk:
                    idn = nat.conv_gemm(t, blk["wd"], taps=1, scale=blk["ad"][0], bias=blk["ad"][1], act=0,
                                        stride=blk["stride"])
                elif not idn.is_contiguous():
                    idn = idn.contiguous()   # (never: a sliced feature is only ever a first-block input)
                out = None
                if last and fi is not None and fi in dest:
                    ci, off, total = dest[fi]
                    if bufs[ci] is None:
                        bufs[ci] = torch.empty((B, h.shape[1], h.shape[2], total), dtype=torch.bfloat16, device=dev)
                    if tuple(bufs[ci].shape[1:3]) != tuple(h.shape[1:3]):
                        raise ValueError("features of one chain must share their spatial size (torch.cat would fail too)")
                    out = bufs[ci][..., off:off + chans[li]]
                t = nat.conv_gemm(h, blk["w3"], taps=1, scale=blk["a3"][0], bias=blk["a3"][1], res=idn, res_mode=1,
                                  act=2, out=out)
            if fi is not None:
                feats.append(t)
        if chains is not None:
            return bufs
        return feats


def build_radimagenet_backbone(name="resnet50", device="cuda", in_channels=6, output_stride=8, out_indices=(1, 2, 3, 4),
                               use_advanced_adapt=True, pretrained_path=None):
    """Reference :220-312 without timm / the checkpoint download (no network): the same ResNet-50 feature extractor;
    `pretrained_path` (a local RadImageNet or timm state dict) is loaded when given, re-keyed as the reference does."""
    if name != "resnet50":
        raise NotImplementedError("RadImageNet ResNet-101 is not built")
    model = B200ResNetBackbone(in_chans=in_channels, output_stride=output_stride, out_indices=out_indices)
    if pretrained_path is not None:
        ckpt = torch.load(pretrained_path, map_location="cpu")
        for key in ("state_dict", "model_state_dict", "model", "encoder"):
            if isinstance(ckpt, dict) and key in ckpt and isinstance(ckpt[key], dict):
                ckpt = ckpt[key]
                break
        ckpt = map_rasool_to_timm_keys(ckpt)
        own = model.state_dict()
        w = ckpt.get("conv1.weight")
        if w is not None and w.shape[1] != in_channels:  # adapt_first_conv (:70-95): mean over RGB, repeated
            ckpt["conv1.weight"] = w.mean(dim=1, keepdim=True).repeat(1, in_channels, 1, 1)
        model.load_state_dict({k: v for k, v in ckpt.items() if k in own and own[k].shape == v.shape}, strict=False)
    model.eval()
    return model.to(device) if device is not None else model


build_imagenet_backbone = build_radimagenet_backbone


def map_rasool_to_timm_keys(rasool_state_dict):
    """Reference :180-218: RadImageNet (Rasool) ResNet-50 keys -> timm resnet50 keys."""
    layer_map = {"4": "layer1", "5": "layer2", "6": "layer3", "7": "layer4"}
    mapped = {}
    for k, v in rasool_state_dict.items():
        nk = k[len("backbone."):] if k.startswith("backbone.") else k
        if nk == "0.weight":
            nk = "conv1.weight"
        elif nk.startswith("1."):
            nk = "bn1." + nk[2:]
        elif nk[:1] in layer_map and nk[1:2] == ".":
            nk = f"{layer_map[nk[0]]}.{nk[2:]}"
        if nk.startswith("fc."):
            continue
        mapped[nk] = v
    return mapped


def build_vit_dino_backbone(model_name="vit_base_patch16_224", in_channels=3, img_size=224, device=None, **_):
    """Reference :371-431 without the timm dependency: a ViT-B/16 feature extractor for `in_channels` inputs."""
    if model_name not in VIT_NAMES:
        raise ValueError(f"unsupported ViT name {model_name!r}")
    size = img_size[0] if isinstance(img_size, (tuple, list)) else img_size
    model = B200ViTBackbone(in_chans=in_channels, img_size=size)
    return model.to(device) if device is not None else model


def build_medical_backbone(parameters, device, method, in_channels):
    """Reference :490-577, ViT branch (:526-545).  Mutates parameters[f"{method}_model_parameters"]."""
    mp = parameters[f"{method}_model_parameters"]
    name = mp["backbone_str"]
    if name in RESNET_NAMES:
        # reference :503-524 (resnet50) and :547-569 (radimagenet): C2 / C3 / C4+C5 chains, block1 down-samples
        backbone = build_radimagenet_backbone("resnet50", device=device, in_channels=in_channels,
                                              output_stride=mp.get("backbone_stride", 8))
        mp["backbone_index_lists"] = [[0], [1], [2, 3]]
        mp["downsample"] = (True, False, False)
        mp["downsample_each_repeat"] = False
        return backbone
    if name not in VIT_NAMES:
        raise NotImplementedError(
            f"backbone {name!r}: only the ViT-B/16 branch is built (ResNet / RadImageNet / UNI2-h need network "
            "access and timm; SURVEY.md section 2)")
    backbone = build_vit_dino_backbone("vit_base_patch16_224", in_channels=in_channels, img_size=mp["input_size"],
                                       device=device)
    mp["backbone_index_lists"] = [[0, 1, 2], [3, 4, 5, 6], [7, 8, 9, 10, 11]]
    mp["downsample"] = (False, False, False)
    mp["channels"] = (backbone.embed_dim,) * 3
    mp["transformer_backbone"] = True
    backbone.eval()
    return backbone
