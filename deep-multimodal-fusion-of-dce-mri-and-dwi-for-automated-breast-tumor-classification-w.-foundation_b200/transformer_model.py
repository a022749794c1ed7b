"""B200-native drop-in for the reference's ``transformer_model`` (code/transformer_model.py).

Same class names, constructor signatures and parameter names as the reference's in-house
pre-norm transformer stage (PatchEmbed :7-32, TokensToFeatureMap :34-52, TransformerEncoder
:54-66, TransformerBlock :68-81, MultiHeadSelfAttention :83-116, MLP :118-134,
TransformerStage :137-175).  Inside ModelMaskHeadBackbone.forward the stage is scheduled as one fused sequence
(model_module._transformer_stage: packed weights cached, LayerScale + residual folded into the GEMM epilogues, fp32
residual stream).  Called on their own, the modules run the same sm_100a kernels in eval mode - linears on
b200_conv_gemm_ex / b200_linear, LayerNorm on b200_layernorm, softmax(q k^T) v on b200_attention - with the reference's
tensor conventions (tokens [B, N, C] fp32 in and out, maps NCHW).  CUDA only; train mode raises (the training path
of the hybrid stage is not built).
"""
from __future__ import annotations

import torch
import torch.nn as nn

__all__ = ["PatchEmbed", "TokensToFeatureMap", "TransformerEncoder", "TransformerBlock", "MultiHeadSelfAttention",
           "MLP", "TransformerStage"]


def _nat(mod, name, x):
    """Guards shared by the stand-alone forwards; returns the native-call module."""
    import b200_native as nat

    if mod.training:
        raise NotImplementedError(f"{name}.forward in training mode is not built: .eval() for the inference forward")
    if not x.is_cuda:
        raise nat.B200NativeError(f"{name}.forward needs a CUDA tensor (no CPU path)")
    return nat


def _w(t):
    return t.detach().to(torch.bfloat16).contiguous()


def _f(t):
    return t.detach().float().contiguous()


def _tokens_bf16(x):
    B, N, C = x.shape
    return x.reshape(B * N, C).to(torch.bfloat16).contiguous()


def _attention_tokens(nat, at, h, B, N):
    """h [B*N, C] bf16 (already normalised) -> proj(softmax(q k^T / sqrt d) v) [B*N, C] bf16 (reference :98-116)."""
    C = at.embed_dim
    if at.head_dim not in (64, 128):
        raise NotImplementedError("b200_attention: head_dim 64 or 128")
    bqkv = _f(at.qkv.bias) if at.qkv.bias is not None else torch.zeros(3 * C, device=h.device)
    qkv = nat.linear(h, _w(at.qkv.weight), bias=bqkv)
    o = torch.empty((B * N, C), dtype=torch.bfloat16, device=h.device)
    nat.attention(qkv, o, B, N, at.num_heads, at.head_dim, scale=at.scale)
    return o


def _block_tokens(nat, blk, t, B, N):
    """One pre-norm block on the fp32 residual stream t [B*N, C] (reference :77-81): LayerScale and the residual
    add ride in the proj / fc2 GEMM epilogues, out = acc * gamma + gamma * bias + t."""
    g1, g2 = _f(blk.gamma1), _f(blk.gamma2)
    h = nat.layernorm(t, _f(blk.norm1.weight), _f(blk.norm1.bias), blk.norm1.eps)
    o = _attention_tokens(nat, blk.attn, h, B, N)
    t2 = nat.linear_f32(o, _w(blk.attn.proj.weight), scale=g1, bias=(g1 * _f(blk.attn.proj.bias)).contiguous(), res=t,
                        res_mode=2, out_dtype=torch.float32)
    h = nat.layernorm(t2, _f(blk.norm2.weight), _f(blk.norm2.bias), blk.norm2.eps)
    u = nat.linear(h, _w(blk.mlp.fc1.weight), bias=_f(blk.mlp.fc1.bias), act=1)
    return nat.linear_f32(u, _w(blk.mlp.fc2.weight), scale=g2, bias=(g2 * _f(blk.mlp.fc2.bias)).contiguous(), res=t2,
                          res_mode=2, out_dtype=torch.float32)


class PatchEmbed(nn.Module):
    def __init__(self, in_ch, embed_dim, patch_size=2, dim=2):
        super().__init__()
        if dim != 2:
            raise NotImplementedError("dim=2 only")
        self.dim = dim
        self.norm = nn.LayerNorm(embed_dim)
        self.proj = nn.Conv2d(in_ch, embed_dim, kernel_size=patch_size, stride=patch_size)

    def forward(self, x):
        """x [B, C, H, W] -> (tokens [B, N, E] fp32, (H/p, W/p)) (reference :26-32): the strided conv as an implicit
        GEMM on b200_conv_gemm_ex (taps = 4), LayerNorm on b200_layernorm."""
        nat = _nat(self, "PatchEmbed", x)
        if self.proj.kernel_size != (2, 2) or self.proj.stride != (2, 2):
            raise NotImplementedError("only patch_size=2 (the reference default) is built")
        import model_module as mm

        xh = mm._as_nhwc_bf16(x)
        tok = nat.conv_gemm(xh, mm._conv_w_bf16(self.proj, x.device), taps=4, bias=_f(self.proj.bias))
        B, Ht, Wt, E = tok.shape
        t = nat.layernorm(tok.view(B * Ht * Wt, E), _f(self.norm.weight), _f(self.norm.bias), self.norm.eps,
                          out_dtype=torch.float32)
        return t.view(B, Ht * Wt, E), (Ht, Wt)


class TokensToFeatureMap(nn.Module):
    def __init__(self, dim=2):
        super().__init__()
        self.dim = dim

    def forward(self, tokens, spatial_shape):
        B, N, C = tokens.shape
        H, W = spatial_shape
        return tokens.transpose(1, 2).reshape(B, C, H, W)  # pure view bookkeeping, no arithmetic


class MultiHeadSelfAttention(nn.Module):
    def __init__(self, embed_dim, num_heads, qkv_bias=True, attn_drop=0.1, proj_drop=0.1):
        super().__init__()
        assert embed_dim % num_heads == 0, "embed_dim must be divisible by num_heads"
        self.embed_dim, self.num_heads = embed_dim, num_heads
        self.head_dim = embed_dim // num_heads
        self.scale = self.head_dim ** -0.5
        self.qkv = nn.Linear(embed_dim, embed_dim * 3, bias=qkv_bias)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(embed_dim, embed_dim)
        self.proj_drop = nn.Dropout(proj_drop)

    def forward(self, x):
        """x [B, N, C] -> [B, N, C] fp32 (reference :98-116; attn_drop / proj_drop are identity in eval mode)."""
        nat = _nat(self, "MultiHeadSelfAttention", x)
        B, N, C = x.shape
        o = _attention_tokens(nat, self, _tokens_bf16(x), B, N)
        y = nat.linear_f32(o, _w(self.proj.weight), bias=_f(self.proj.bias), out_dtype=torch.float32)
        return y.view(B, N, C)


class MLP(nn.Module):
    def __init__(self, embed_dim, mlp_ratio=4.0, drop=0.1):
        super().__init__()
        hidden = int(embed_dim * mlp_ratio)
        self.fc1 = nn.Linear(embed_dim, hidden)
        self.act = nn.GELU()
        self.fc2 = nn.Linear(hidden, embed_dim)
        self.drop = nn.Dropout(drop)

    def forward(self, x):
        """x [B, N, C] -> fc2(gelu(fc1 x)) fp32 (reference :128-134), both GEMMs on the tcgen05 kernel."""
        nat = _nat(self, "MLP", x)
        B, N, C = x.shape
        u = nat.linear(_tokens_bf16(x), _w(self.fc1.weight), bias=_f(self.fc1.bias), act=1)
        return nat.linear_f32(u, _w(self.fc2.weight), bias=_f(self.fc2.bias), out_dtype=torch.float32).view(B, N, C)


class TransformerBlock(nn.Module):
    def __init__(self, embed_dim, heads, init_scale=0.1):
        super().__init__()
        self.norm1 = nn.LayerNorm(embed_dim)
        self.attn = MultiHeadSelfAttention(embed_dim, heads)
        self.norm2 = nn.LayerNorm(embed_dim)
        self.mlp = MLP(embed_dim)
        self.gamma1 = nn.Parameter(init_scale * torch.ones(embed_dim))
        self.gamma2 = nn.Parameter(init_scale * torch.ones(embed_dim))

    def forward(self, x):
        """x [B, N, C] -> x + gamma1 * attn(norm1 x), then + gamma2 * mlp(norm2 .) (reference :77-81), fp32 stream."""
        nat = _nat(self, "TransformerBlock", x)
        B, N, C = x.shape
        return _block_tokens(nat, self, x.reshape(B * N, C).float().contiguous(), B, N).view(B, N, C)


class TransformerEncoder(nn.Module):
    def __init__(self, embed_dim, depth=4, heads=8):
        super().__init__()
        self.layers = nn.ModuleList([TransformerBlock(embed_dim, heads=heads) for _ in range(depth)])

    def forward(self, x):
        nat = _nat(self, "TransformerEncoder", x)
        B, N, C = x.shape
        t = x.reshape(B * N, C).float().contiguous()
        for layer in self.layers:
            t = _block_tokens(nat, layer, t, B, N)
        return t.view(B, N, C)


class TransformerStage(nn.Module):
    def __init__(self, in_ch, embed_dim, depth=2, heads=8, patch_size=2, dim=2):
        super().__init__()
        if dim != 2:
            raise NotImplementedError("dim=2 only")
        self.dim = dim
        self.patch_embed = PatchEmbed(in_ch=in_ch, embed_dim=embed_dim, patch_size=patch_size, dim=dim)
        self.transformer = TransformerEncoder(embed_dim=embed_dim, depth=depth, heads=heads)
        self.tokens_to_map = TokensToFeatureMap(dim=dim)

    def forward(self, x):
        """x [B, C, H, W] -> [B, E, H/p, W/p] (reference :170-175)."""
        _nat(self, "TransformerStage", x)
        tokens, spatial_shape = self.patch_embed(x)
        return self.tokens_to_map(self.transformer(tokens), spatial_shape)
