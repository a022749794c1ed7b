"""Kernel-level numerics on the GPU: every C-ABI op against a plain PyTorch fp32 restatement
of the same op on the same (bf16-rounded) operands.  Tolerances are stated per test."""
import math

import pytest
import torch
import torch.nn.functional as F

import b200_native as nat

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _rel(a, b):
    return (a.float() - b.float()).abs().max().item() / max(b.float().abs().max().item(), 1e-12)


def _conv_ref(x, w, taps, scale, bias, res, res_mode, act):
    B, H, W, Cin = x.shape
    Cout = w.shape[0]
    xf = x.float().permute(0, 3, 1, 2)
    k = 3 if taps == 9 else 1
    wf = w.float().view(Cout, taps, Cin).permute(0, 2, 1).reshape(Cout, Cin, k, k)
    y = F.conv2d(xf, wf, padding=k // 2)
    if scale is not None:
        y = y * scale.view(1, -1, 1, 1)
    if bias is not None:
        y = y + bias.view(1, -1, 1, 1)
    r = res.float().permute(0, 3, 1, 2) if res is not None else None
    if res_mode == 1:
        y = y + r
    if act:
        y = F.gelu(y)
    if res_mode == 2:
        y = y + r
    return y.permute(0, 2, 3, 1).contiguous()


@pytest.mark.parametrize("B,H,W,Cin,Cout,taps,res_mode,act,gap,up2", [
    (2, 32, 32, 64, 64, 1, 0, 0, False, False),
    (2, 32, 32, 64, 64, 9, 0, 1, False, False),
    (3, 32, 32, 64, 128, 1, 1, 1, True, False),
    (2, 32, 32, 128, 128, 9, 0, 1, False, False),
    (2, 32, 32, 128, 256, 1, 2, 1, False, False),
    (5, 32, 32, 256, 256, 9, 0, 1, True, False),
    (2, 32, 32, 256, 512, 1, 1, 1, True, False),
    (2, 32, 32, 128, 64, 1, 0, 1, False, True),
    (1, 64, 64, 64, 64, 9, 0, 1, False, False),
    (40, 32, 32, 256, 256, 9, 0, 1, True, False),   # > 148 tiles: persistent loop + both TMEM stages
])
def test_conv_gemm(B, H, W, Cin, Cout, taps, res_mode, act, gap, up2):
    g = torch.Generator(device="cpu").manual_seed(B * 1000 + Cin + Cout + taps)
    x = (torch.randn(B, H, W, Cin, generator=g) * 0.5).to(DEV).bfloat16()
    w = (torch.randn(Cout, taps * Cin, generator=g) / math.sqrt(taps * Cin)).to(DEV).bfloat16()
    scale = (torch.rand(Cout, generator=g) + 0.5).to(DEV)
    bias = (torch.randn(Cout, generator=g) * 0.1).to(DEV)
    res = (torch.randn(B, H, W, Cout, generator=g) * 0.5).to(DEV).bfloat16() if res_mode else None
    gap_buf = torch.zeros(B, Cout, device=DEV) if gap else None
    y = nat.conv_gemm(x, w, taps=taps, scale=scale, bias=bias, res=res, res_mode=res_mode, act=act, gap=gap_buf,
                      up2=up2)
    torch.cuda.synchronize()
    ref = _conv_ref(x, w, taps, scale, bias, res, res_mode, act)
    if up2:
        ref = ref.repeat_interleave(2, dim=1).repeat_interleave(2, dim=2)
    # bf16 output rounding: 2^-9 relative per element; accumulation is fp32
    assert _rel(y, ref) < 1e-2
    assert (y.float() - ref).abs().max().item() < 2e-2 * max(1.0, ref.abs().max().item())
    if gap:
        gref = _conv_ref(x, w, taps, scale, bias, res, res_mode, act).sum(dim=(1, 2))
        assert _rel(gap_buf, gref) < 1e-3


@pytest.mark.parametrize("M,K,N", [(197, 768, 768), (1000, 128, 64), (128, 64, 256), (77, 3072, 768)])
def test_linear_ragged_rows(M, K, N):
    g = torch.Generator(device="cpu").manual_seed(M + K + N)
    x = (torch.randn(M, K, generator=g) * 0.5).to(DEV).bfloat16()
    w = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(DEV).bfloat16()
    bias = (torch.randn(N, generator=g) * 0.1).to(DEV)
    y = nat.linear(x, w, bias=bias, act=1)
    torch.cuda.synchronize()
    ref = F.gelu(x.float() @ w.float().t() + bias)
    assert _rel(y, ref) < 1e-2


@pytest.mark.parametrize("B,Cin,n1,n2", [(3, 128, 256, 128), (2, 256, 512, 256), (2, 64, 64, 64)])
def test_conv_gemm_two_segments(B, Cin, n1, n2):
    """Skip conv (no activation) and first bottleneck conv (GELU) on the same input in one launch."""
    g = torch.Generator(device="cpu").manual_seed(Cin + n1)
    x = (torch.randn(B, 32, 32, Cin, generator=g) * 0.5).to(DEV).bfloat16()
    w = (torch.randn(n1 + n2, Cin, generator=g) / math.sqrt(Cin)).to(DEV).bfloat16()
    scale = (torch.rand(n1 + n2, generator=g) + 0.5).to(DEV)
    bias = (torch.randn(n1 + n2, generator=g) * 0.1).to(DEV)
    y1, y2 = nat.conv_gemm(x, w, taps=1, scale=scale, bias=bias, act=0, n_split=n1, act2=1)
    torch.cuda.synchronize()
    ref = _conv_ref(x, w, 1, scale, bias, None, 0, 0)
    assert y1.shape[-1] == n1 and y2.shape[-1] == n2
    assert _rel(y1, ref[..., :n1]) < 1e-2
    assert _rel(y2, F.gelu(ref[..., n1:])) < 1e-2


@pytest.mark.parametrize("B,C", [(2, 128), (3, 256), (1, 64)])
def test_recon_head_fused_tap_dots(B, C):
    """3x3 conv + affine + GELU with the following 3x3, C->1 conv folded into the epilogue + tapsum."""
    g = torch.Generator(device="cpu").manual_seed(C)
    x = (torch.randn(B, 32, 32, C, generator=g) * 0.5).to(DEV).bfloat16()
    w = (torch.randn(C, 9 * C, generator=g) / math.sqrt(9 * C)).to(DEV).bfloat16()
    scale = (torch.rand(C, generator=g) + 0.5).to(DEV)
    bias = (torch.randn(C, generator=g) * 0.1).to(DEV)
    w3 = (torch.randn(9, C, generator=g) / math.sqrt(9 * C)).to(DEV)
    b3 = torch.tensor([0.3], device=DEV)
    d = torch.empty(B, 32, 32, 9, device=DEV)
    nat.conv_gemm(x, w, taps=9, scale=scale, bias=bias, act=1, store=False, dot_w=w3, dot_out=d)
    out = nat.tapsum(d, b3, torch.empty(B, 32, 32, device=DEV))
    torch.cuda.synchronize()
    t = _conv_ref(x, w, 9, scale, bias, None, 0, 1)  # fp32, not rounded to bf16 (the fused path keeps fp32 too)
    ref = F.conv2d(t.permute(0, 3, 1, 2), w3.view(9, C).t().reshape(1, C, 3, 3), b3, padding=1)[:, 0]
    assert _rel(out, ref) < 5e-3
    # and the stand-alone N=1 kernel on a bf16 map agrees with torch as well
    tb = t.bfloat16()
    out2 = nat.conv3x3_c1(tb, w3, b3, torch.empty(B, 32, 32, device=DEV))
    ref2 = F.conv2d(tb.float().permute(0, 3, 1, 2), w3.view(9, C).t().reshape(1, C, 3, 3), b3, padding=1)[:, 0]
    assert _rel(out2, ref2) < 1e-3


def test_fast_gelu_deviation_from_erf_gelu():
    """The epilogue GELU is 0.5 x (1 + tanh(x (c0 + c1 x^2))) on MUFU.TANH (common.cuh gelu_fast2): compared with
    nn.GELU()'s erf form through an identity 1x1 'convolution' (weights = I) over [-9, 9].  Bound: the bf16 rounding of
    the output (4e-3 relative) plus 1.2e-3 absolute (4.7e-4 from the tanh form, the rest from MUFU.TANH's 2^-11
    relative error on 1 + tanh); exact zero / identity far from the origin."""
    C = 64
    xs = torch.linspace(-9, 9, 2 * 32 * 32 * C).view(2, 32, 32, C).to(DEV).bfloat16()
    w = torch.eye(C, device=DEV).bfloat16()
    y = nat.conv_gemm(xs, w, taps=1, act=1)
    torch.cuda.synchronize()
    ref = F.gelu(xs.float())
    err = (y.float() - ref).abs()
    print("fast GELU: max |d| =", err.max().item(), "at x =", xs.float().flatten()[err.argmax()].item())
    assert (err <= 4e-3 * ref.abs() + 1.2e-3).all(), err.max()
    far = xs.float().abs() > 6.5
    assert (err[far] <= 4e-3 * ref[far].abs() + 2e-4).all(), err[far].max()   # saturated: 0 or x, no tanh residue


def test_fused_single_dot_is_a_following_1x1_conv_to_one_channel():
    """Mask head: `pre` 1x1 conv + bias with `out` (C -> 1) folded into the epilogue (ndot = 1)."""
    g = torch.Generator(device="cpu").manual_seed(3)
    B, Cin, C = 3, 256, 64
    x = (torch.randn(B, 32, 32, Cin, generator=g) * 0.5).to(DEV).bfloat16()
    w = (torch.randn(C, Cin, generator=g) / math.sqrt(Cin)).to(DEV).bfloat16()
    bias = (torch.randn(C, generator=g) * 0.1).to(DEV)
    wo = (torch.randn(1, C, generator=g) / math.sqrt(C)).to(DEV)
    out = torch.empty(B, 32, 32, 1, device=DEV)
    nat.conv_gemm(x, w, taps=1, bias=bias, store=False, dot_w=wo, dot_out=out, dot_bias=0.25)
    torch.cuda.synchronize()
    ref = (x.float() @ w.float().t() + bias) @ wo.t() + 0.25
    assert _rel(out, ref) < 1e-4


def test_patch_embed_conv_2x2_stride2():
    """PatchEmbed.proj (transformer_model.py:18-23): 2x2 kernel, stride 2, bias -> tokens."""
    g = torch.Generator(device="cpu").manual_seed(8)
    B, Cin, Cout = 3, 256, 512
    x = (torch.randn(B, 32, 32, Cin, generator=g) * 0.5).to(DEV).bfloat16()
    w4 = (torch.randn(Cout, Cin, 2, 2, generator=g) / math.sqrt(4 * Cin)).to(DEV)
    bias = (torch.randn(Cout, generator=g) * 0.1).to(DEV)
    w = w4.permute(0, 2, 3, 1).reshape(Cout, -1).bfloat16().contiguous()
    y = nat.conv_gemm(x, w, taps=4, bias=bias)
    torch.cuda.synchronize()
    assert tuple(y.shape) == (B, 16, 16, Cout)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), w4.bfloat16().float(), bias, stride=2).permute(0, 2, 3, 1)
    assert _rel(y, ref) < 1e-2


@pytest.mark.parametrize("C", [256, 512, 768])
def test_layernorm(C):
    g = torch.Generator(device="cpu").manual_seed(C)
    x = (torch.randn(1000, C, generator=g) * 2 + 0.3).to(DEV).bfloat16()
    w = (torch.rand(C, generator=g) + 0.5).to(DEV)
    b = (torch.randn(C, generator=g) * 0.1).to(DEV)
    y = nat.layernorm(x, w, b, 1e-5)
    y32 = nat.layernorm(x.float(), w, b, 1e-5, out_dtype=torch.float32)
    torch.cuda.synchronize()
    ref = F.layer_norm(x.float(), (C,), w, b, 1e-5)
    assert _rel(y, ref) < 6e-3  # one bf16 rounding of the output
    assert _rel(y32, ref) < 1e-5


@pytest.mark.parametrize("B,H,W,Hc", [(3, 32, 32, 32), (2, 15, 17, 7)])
def test_mask_attention(B, H, W, Hc):
    """b200_mask_attention: MaskGuidedSpatialAttention.mask_processor (model_module.py:67-73, :92-93) - 1x1 1->Hc,
    GroupNorm(1, Hc), GELU, 1x1 Hc->1, sigmoid, clamp to [1e-4, 1 - 1e-4] - against fp64 torch with nn.GELU()'s erf
    form.  255 pixels is not a multiple of the 256 threads; an odd Hc takes the single-channel tail.  Bound: the
    kernel's GELU is the tanh form (gelu_fast2) on the channel pairs, within 1.2e-3 of erf's
    (test_fast_gelu_deviation_from_erf_gelu), and the exact erf form on the odd tail channel, so the bound is loose
    there; the pre-sigmoid sum is within 1.2e-3 * sum |wb|, and the sigmoid's slope is at most 1/4; 1e-5 for fp32
    rounding."""
    g = torch.Generator(device="cpu").manual_seed(B * 100 + Hc)
    m = torch.randn(B, 1, H, W, generator=g) * 2 + 0.5
    wa = torch.randn(Hc, generator=g)
    gn_w = torch.rand(Hc, generator=g) + 0.5
    gn_b = torch.randn(Hc, generator=g) * 0.2
    wb = torch.randn(Hc, generator=g) / math.sqrt(Hc)
    bb = torch.randn(1, generator=g) * 0.2
    eps = 1e-5
    attn = torch.empty(B, 1, H, W, device=DEV)
    nat.mask_attention(m.to(DEV), (Hc, wa.to(DEV), gn_w.to(DEV), gn_b.to(DEV), wb.to(DEV), bb.to(DEV), eps), attn)
    torch.cuda.synchronize()
    u = F.group_norm(m.double() * wa.double().view(1, Hc, 1, 1), 1, gn_w.double(), gn_b.double(), eps)
    a = (F.gelu(u) * wb.double().view(1, Hc, 1, 1)).sum(1, keepdim=True) + bb.double()
    ref = torch.sigmoid(a).clamp(1e-4, 1 - 1e-4)
    err = (attn.cpu().double() - ref).abs().max().item()
    assert err <= 0.25 * 1.2e-3 * wb.abs().sum().item() + 1e-5, err


@pytest.mark.parametrize("B,heads,N,dh,pad", [(3, 12, 197, 64, 0), (2, 4, 256, 128, 0), (2, 2, 70, 64, 64),
                                              (5, 3, 129, 64, 0), (1, 2, 16, 128, 8), (40, 12, 197, 64, 0)])
def test_fused_attention(B, heads, N, dh, pad):
    """b200_attention: softmax(q k^T / sqrt d) v per (case, head) straight from the packed qkv rows
    (transformer_model.py:101-112), against fp32 torch on the same bf16 inputs.  Covers the ViT-B/16 shape (197 tokens:
    a ragged second query tile and a ragged last key chunk), the hybrid stage (256 x 128), token counts below one
    tile, padded leading dimensions, and more work items than resident CTAs (the persistent loop)."""
    g = torch.Generator(device="cpu").manual_seed(B * heads + N)
    C = heads * dh
    buf = torch.full((B * N, 3 * C + pad), float("nan")).bfloat16().to(DEV)  # NaN padding: must never be read as data
    qkv = buf[:, :3 * C]
    qkv.copy_((torch.randn(B * N, 3 * C, generator=g) * 0.9).bfloat16())
    out_buf = torch.zeros(B * N, C + pad, device=DEV, dtype=torch.bfloat16)
    out = out_buf[:, :C]
    nat.attention(qkv, out, B, N, heads, dh)
    torch.cuda.synchronize()
    q, k, v = (qkv.float().view(B, N, 3, heads, dh).permute(2, 0, 3, 1, 4)[i] for i in range(3))
    ref = (torch.softmax(q @ k.transpose(-1, -2) * dh ** -0.5, dim=-1) @ v).permute(0, 2, 1, 3).reshape(B * N, C)
    assert torch.isfinite(out.float()).all()
    assert _rel(out, ref) < 1.2e-2
    if pad:
        assert torch.count_nonzero(out_buf[:, C:]) == 0


def test_fused_attention_steep_rows_take_the_two_pass_path():
    """The single-read softmax measures exponents against the max of a row's first 32 scores; rows whose later scores
    exceed that by more than ~2^100 overflow the lazy reference and are redone with the row max.  Logits with a
    standard deviation of ~36 (near one-hot rows) exercise that path; the ordinary cases of the same launch do not."""
    g = torch.Generator(device="cpu").manual_seed(77)
    B, heads, N, dh = 4, 12, 197, 64
    C = heads * dh
    x = torch.randn(B * N, 3 * C, generator=g)
    x[: 2 * N, : 2 * C] *= 6.0          # cases 0-1: steep; cases 2-3: ordinary
    x[2 * N:] *= 0.9
    qkv = x.bfloat16().to(DEV)
    out = torch.empty(B * N, C, device=DEV, dtype=torch.bfloat16)
    nat.attention(qkv, out, B, N, heads, dh)
    torch.cuda.synchronize()
    q, k, v = (qkv.float().view(B, N, 3, heads, dh).permute(2, 0, 3, 1, 4)[i] for i in range(3))
    s = q @ k.transpose(-1, -2) * dh ** -0.5
    assert ((s[:2].amax(-1) - s[:2, ..., :32].amax(-1)) * 1.4427 > 128).any()  # the overflow case is really present
    ref = (torch.softmax(s, dim=-1) @ v).permute(0, 2, 1, 3).reshape(B * N, C)
    assert torch.isfinite(out.float()).all()
    assert _rel(out, ref) < 1.2e-2


def test_linear_fp32_residual_stream():
    """x + gamma * (W y + b) with the residual read and the result written in fp32 (transformer blocks)."""
    g = torch.Generator(device="cpu").manual_seed(21)
    M, K, N = 1000, 2048, 512
    y = (torch.randn(M, K, generator=g) * 0.5).to(DEV).bfloat16()
    w = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(DEV).bfloat16()
    gamma = (0.1 * (1 + 0.1 * torch.randn(N, generator=g))).to(DEV)
    bias = (torch.randn(N, generator=g) * 0.1).to(DEV)
    x = torch.randn(M, N, generator=g).to(DEV)
    out = nat.linear_f32(y, w, scale=gamma, bias=gamma * bias, res=x, res_mode=2, out_dtype=torch.float32)
    out_b = nat.linear_f32(y, w, scale=gamma, bias=gamma * bias, res=x, res_mode=2, out_dtype=torch.bfloat16)
    torch.cuda.synchronize()
    ref = x + gamma * (y.float() @ w.float().t() + bias)
    assert out.dtype == torch.float32 and _rel(out, ref) < 1e-5
    assert _rel(out_b, ref) < 6e-3


# ------------------------------------------------------------------ 14 x 14 maps (ViT grid) ----
@pytest.mark.parametrize("B,H,W,Cin,Cout,taps,res_mode,act", [
    (2, 14, 14, 64, 64, 1, 0, 0),
    (3, 14, 14, 128, 256, 9, 0, 1),
    (2, 14, 14, 768, 768, 1, 1, 1),      # block tail: 1x1 + residual + GELU, 3 N tiles
    (2, 14, 14, 2304, 768, 9, 0, 1),     # neck conv on 3 concatenated ViT maps (K = 20 736)
    (90, 14, 14, 384, 384, 9, 0, 1),     # > 148 tiles
    (2, 10, 10, 64, 128, 9, 2, 1),       # 10 x 12-row tiles (120 rows used), single ragged tile per case
    (2, 20, 24, 64, 64, 9, 0, 1),        # 24 x 5 tiles, 4 per case
])
def test_conv_gemm_ragged_tiles(B, H, W, Cin, Cout, taps, res_mode, act):
    """Maps whose width does not divide 128: BW x floor(128/BW) tiles, unused MMA rows masked, direct stores."""
    g = torch.Generator(device="cpu").manual_seed(B + H * 7 + Cin + Cout + taps)
    x = (torch.randn(B, H, W, Cin, generator=g) * 0.5).to(DEV).bfloat16()
    w = (torch.randn(Cout, taps * Cin, generator=g) / math.sqrt(taps * Cin)).to(DEV).bfloat16()
    scale = (torch.rand(Cout, generator=g) + 0.5).to(DEV)
    bias = (torch.randn(Cout, generator=g) * 0.1).to(DEV)
    res = (torch.randn(B, H, W, Cout, generator=g) * 0.5).to(DEV).bfloat16() if res_mode else None
    y = torch.full((B, H, W, Cout), 7.0, device=DEV, dtype=torch.bfloat16)
    nat.conv_gemm(x, w, taps=taps, scale=scale, bias=bias, res=res, res_mode=res_mode, act=act, out=y)
    torch.cuda.synchronize()
    ref = _conv_ref(x, w, taps, scale, bias, res, res_mode, act)
    assert _rel(y, ref) < 1e-2
    with pytest.raises(nat.B200NativeError):  # fused pooling needs staged tiles
        nat.conv_gemm(x, w, taps=taps, scale=scale, bias=bias, gap=torch.zeros(B, Cout, device=DEV))


def test_ragged_tiles_two_segments_and_dots():
    g = torch.Generator(device="cpu").manual_seed(14)
    B, C = 3, 128
    x = (torch.randn(B, 14, 14, C, generator=g) * 0.5).to(DEV).bfloat16()
    w = (torch.randn(256 + 128, C, generator=g) / math.sqrt(C)).to(DEV).bfloat16()
    scale = (torch.rand(384, generator=g) + 0.5).to(DEV)
    bias = (torch.randn(384, generator=g) * 0.1).to(DEV)
    y1, y2 = nat.conv_gemm(x, w, taps=1, scale=scale, bias=bias, act=0, n_split=256, act2=1)
    ref = _conv_ref(x, w, 1, scale, bias, None, 0, 0)
    assert _rel(y1, ref[..., :256]) < 1e-2 and _rel(y2, F.gelu(ref[..., 256:])) < 1e-2
    # recon head (3x3 + GELU, then 3x3 C->1 folded in) on a 14 x 14 map
    w9 = (torch.randn(C, 9 * C, generator=g) / math.sqrt(9 * C)).to(DEV).bfloat16()
    w3 = (torch.randn(9, C, generator=g) / math.sqrt(9 * C)).to(DEV)
    b3 = torch.tensor([0.3], device=DEV)
    d = torch.empty(B, 14, 14, 9, device=DEV)
    nat.conv_gemm(x, w9, taps=9, scale=scale[:C], bias=bias[:C], act=1, store=False, dot_w=w3, dot_out=d)
    out = nat.tapsum(d, b3, torch.empty(B, 14, 14, device=DEV))
    torch.cuda.synchronize()
    t = _conv_ref(x, w9, 9, scale[:C], bias[:C], None, 0, 1)
    ref = F.conv2d(t.permute(0, 3, 1, 2), w3.view(9, C).t().reshape(1, C, 3, 3), b3, padding=1)[:, 0]
    assert _rel(out, ref) < 5e-3


@pytest.mark.parametrize("B,H,W,C", [(3, 14, 14, 768), (2, 32, 32, 128), (5, 7, 9, 72)])
def test_channel_sums_mix_instnorm_add(B, H, W, C):
    g = torch.Generator(device="cpu").manual_seed(C + H)
    a = (torch.randn(B, H, W, C, generator=g) * 0.7 + 0.2).to(DEV).bfloat16()
    b = (torch.randn(B, H, W, C, generator=g) * 0.4 - 0.1).to(DEV).bfloat16()
    s = nat.channel_sums(a)
    assert _rel(s, a.float().sum(dim=(1, 2))) < 1e-5
    # channel slice of a wider buffer (row stride > C)
    if C % 16 == 0:
        s2 = nat.channel_sums(a[..., C // 2:])
        assert _rel(s2, a[..., C // 2:].float().sum(dim=(1, 2))) < 1e-5
    wl = torch.tensor([0.3], device=DEV)
    gw = (torch.rand(C, generator=g) + 0.5).to(DEV)
    gb = (torch.randn(C, generator=g) * 0.1).to(DEV)
    y = nat.mix_instnorm(a, b, wl, gw, gb, 1e-5)
    al = torch.sigmoid(wl)
    m = (al * a.float() + (1 - al) * b.float()).permute(0, 3, 1, 2)
    ref = F.group_norm(m, C, gw, gb, 1e-5).permute(0, 2, 3, 1)
    assert _rel(y, ref) < 1e-2          # bf16 output rounding
    z = nat.add_maps(a, b)
    torch.cuda.synchronize()
    assert _rel(z, a.float() + b.float()) < 1e-2


@pytest.mark.parametrize("H,size,C", [(14, 64, 64), (32, 64, 64), (14, 4, 128), (64, 64, 8)])
def test_adaptive_pool(H, size, C):
    g = torch.Generator(device="cpu").manual_seed(H + size)
    x = (torch.randn(2, H, H, C, generator=g)).to(DEV).bfloat16()
    ref = F.adaptive_avg_pool2d(x.float().permute(0, 3, 1, 2), (size, size)).permute(0, 2, 3, 1)
    assert _rel(nat.adaptive_pool(x, size), ref) < 1e-2
    assert _rel(nat.adaptive_pool(x, size, act=1), F.gelu(ref)) < 1e-2
    r = torch.randn(3, H, H, generator=g).to(DEV)
    ref1 = F.adaptive_avg_pool2d(r.unsqueeze(1), (size, size))[:, 0]
    out1 = nat.adaptive_pool(r, size)
    torch.cuda.synchronize()
    assert _rel(out1, ref1) < 1e-6


def test_patchify_gate_and_feature_slices():
    g = torch.Generator(device="cpu").manual_seed(3)
    B, C, P, E, n = 2, 6, 16, 768, 196
    x = torch.rand(B, C, 224, 224, generator=g).to(DEV)
    gate = torch.rand(B, C, generator=g).to(DEV)
    out = torch.empty(B * n, C * P * P, dtype=torch.bfloat16, device=DEV)
    nat.patchify(x, P, out, gate)
    ref = F.unfold(x * gate.view(B, C, 1, 1), P, stride=P).transpose(1, 2).reshape(B * n, -1)
    assert _rel(out, ref) < 5e-3
    t = torch.randn(B, n + 1, E, generator=g).to(DEV)
    buf = torch.zeros(B, 14, 14, 3 * E, dtype=torch.bfloat16, device=DEV)
    nat.vit_feature(t, B, n, E, buf[..., E:2 * E], out_ld=3 * E)
    torch.cuda.synchronize()
    assert _rel(buf[..., E:2 * E].reshape(B, n, E), t[:, 1:]) < 5e-3
    assert buf[..., :E].abs().max().item() == 0 and buf[..., 2 * E:].abs().max().item() == 0


@pytest.mark.parametrize("B,C,Cm", [(256, 768, 384), (37, 128, 64), (5, 16, 8), (3, 6, 3)])
def test_se_gate(B, C, Cm):
    g = torch.Generator(device="cpu").manual_seed(B + C)
    gap = (torch.randn(B, C, generator=g) * 50).to(DEV)
    w1 = (torch.randn(Cm, C, generator=g) / math.sqrt(C)).to(DEV)
    b1 = (torch.randn(Cm, generator=g) * 0.1).to(DEV)
    w2 = (torch.randn(C, Cm, generator=g) / math.sqrt(Cm)).to(DEV)
    b2 = (torch.randn(C, generator=g) * 0.1).to(DEV)
    gate = torch.empty(B, C, device=DEV)
    nat.se_gate(gap, 196, w1.t().contiguous(), b1, w2.t().contiguous(), b2, gate)
    torch.cuda.synchronize()
    ref = torch.sigmoid(F.linear(F.gelu(F.linear(gap / 196, w1, b1)), w2, b2))
    assert _rel(gate, ref) < 1e-5


@pytest.mark.parametrize("B,H,W,Cin,Cout,taps", [(3, 64, 64, 64, 64, 9), (2, 128, 128, 64, 64, 9), (2, 32, 32, 128, 256, 1),
                                                 (2, 64, 64, 64, 128, 1)])
def test_conv_gemm_stride2(B, H, W, Cin, Cout, taps):
    """Strided 3x3 (padding 1) and 1x1 convolutions through the TMA traversal stride (mask-head stacks, stride-2 blocks)."""
    g = torch.Generator(device="cpu").manual_seed(H + Cin + taps)
    x = (torch.randn(B, H, W, Cin, generator=g) * 0.5).to(DEV).bfloat16()
    w = (torch.randn(Cout, taps * Cin, generator=g) / math.sqrt(taps * Cin)).to(DEV).bfloat16()
    bias = (torch.randn(Cout, generator=g) * 0.1).to(DEV)
    y = nat.conv_gemm(x, w, taps=taps, bias=bias, act=1, stride=2)
    torch.cuda.synchronize()
    k = 3 if taps == 9 else 1
    wf = w.float().view(Cout, taps, Cin).permute(0, 2, 1).reshape(Cout, Cin, k, k)
    ref = F.gelu(F.conv2d(x.float().permute(0, 3, 1, 2), wf, bias, stride=2, padding=k // 2)).permute(0, 2, 3, 1)
    assert tuple(y.shape) == (B, H // 2, W // 2, Cout)
    assert _rel(y, ref) < 1e-2


def test_mc_dropout_epilogue_properties():
    """Philox dropout in the GEMM epilogue: survivors are the undropped values x 1/(1-p), the drop rate is p, the
    decisions depend on the seed only, segment selection and the fused channel sums follow the dropped map."""
    g = torch.Generator(device="cpu").manual_seed(77)
    B, H, W, Cin, n1, n2, p = 4, 32, 32, 128, 128, 128, 0.2
    x = (torch.randn(B, H, W, Cin, generator=g) * 0.5).to(DEV).bfloat16()
    w = (torch.randn(n1 + n2, Cin, generator=g) / math.sqrt(Cin)).to(DEV).bfloat16()
    bias = (torch.randn(n1 + n2, generator=g) * 0.1 + 1.0).to(DEV)   # keeps outputs away from 0
    a1, a2 = nat.conv_gemm(x, w, taps=1, bias=bias, act=0, n_split=n1, act2=1)
    d1, d2 = nat.conv_gemm(x, w, taps=1, bias=bias, act=0, n_split=n1, act2=1, dropout=(p, 1234, 2))
    e1, e2 = nat.conv_gemm(x, w, taps=1, bias=bias, act=0, n_split=n1, act2=1, dropout=(p, 1234, 2))
    f1, f2 = nat.conv_gemm(x, w, taps=1, bias=bias, act=0, n_split=n1, act2=1, dropout=(p, 99, 2))
    z1, _ = nat.conv_gemm(x, w, taps=1, bias=bias, act=0, n_split=n1, act2=1)   # the request is one-shot
    torch.cuda.synchronize()
    assert torch.equal(a1, d1) and torch.equal(a1, z1)       # segment 1 untouched
    assert torch.equal(d2, e2) and not torch.equal(d2, f2)   # same seed -> same mask; other seed -> other mask
    dropped = d2 == 0
    rate = dropped.float().mean().item()
    n = d2.numel()
    assert abs(rate - p) < 5 * math.sqrt(p * (1 - p) / n) + 1e-3
    keep = ~dropped
    assert _rel(d2[keep], a2[keep].float() / (1 - p)) < 1e-2
    # no structure along channels / pixels: per-channel and per-pixel drop rates stay near p
    assert (dropped.float().mean(dim=(0, 1, 2)) - p).abs().max().item() < 0.03
    assert (dropped.float().mean(dim=3) - p).abs().max().item() < 0.2
    # residual + GELU + fused channel sums on a dropped map
    res = (torch.randn(B, H, W, 256, generator=g) * 0.5 + 1.0).to(DEV).bfloat16()
    gap = torch.zeros(B, 256, device=DEV)
    y = nat.conv_gemm(x, w, taps=1, bias=bias, res=res, res_mode=1, act=1, gap=gap, dropout=(0.5, 7, 1))
    torch.cuda.synchronize()
    assert abs((y == 0).float().mean().item() - 0.5) < 0.01
    assert _rel(gap, y.float().sum(dim=(1, 2))) < 1e-3


def test_flip_planes():
    x = torch.randn(5, 6, 24, 40, device=DEV)
    assert torch.equal(nat.flip_planes(x, True, False), torch.flip(x, dims=[-1]))
    assert torch.equal(nat.flip_planes(x, False, True), torch.flip(x, dims=[-2]))
    assert torch.equal(nat.flip_planes(x, True, True), torch.flip(x, dims=[-1, -2]))


def test_resnet_gemm_stem_and_dilated_relu_conv():
    g = torch.Generator(device="cpu").manual_seed(9)
    x = torch.rand(3, 6, 64, 80, generator=g).to(DEV)
    gate = (torch.rand(3, 6, generator=g) + 0.5).to(DEV)
    w = (torch.randn(64, 6, 7, 7, generator=g) / math.sqrt(6 * 49)).to(DEV)
    scale = (torch.rand(64, generator=g) + 0.5).to(DEV)
    bias = (torch.randn(64, generator=g) * 0.1).to(DEV)
    # the stem as B200ResNetBackbone runs it: bf16 im2col rows (gate applied) and one GEMM with the folded BN + ReLU
    kp = (6 * 49 + 63) // 64 * 64
    wg = torch.zeros(64, kp, dtype=torch.bfloat16, device=DEV)
    wg[:, :6 * 49] = w.flatten(1).bfloat16()
    y = nat.linear(nat.im2col7x7_s2(x, gate, kp), wg, scale=scale, bias=bias, act=2).view(3, 32, 40, 64)
    # reference on the bf16-rounded operands: only the accumulation order and the output rounding differ
    xg = (x * gate.view(3, 6, 1, 1)).bfloat16().float()
    ref = F.relu(F.conv2d(xg, w.bfloat16().float(), stride=2, padding=3) * scale.view(1, -1, 1, 1) +
                 bias.view(1, -1, 1, 1)).permute(0, 2, 3, 1)
    assert _rel(y, ref) < 5e-3
    p = nat.maxpool3x3_s2(y)
    refp = F.max_pool2d(y.float().permute(0, 3, 1, 2), 3, stride=2, padding=1).permute(0, 2, 3, 1)
    assert torch.equal(p.float(), refp)
    # dilated 3x3 + ReLU on a 28 x 28 map (ragged 112-row tiles), residual + ReLU on a channel slice
    a = (torch.randn(2, 28, 28, 128, generator=g) * 0.5).to(DEV).bfloat16()
    w3 = (torch.randn(128, 9 * 128, generator=g) / math.sqrt(9 * 128)).to(DEV).bfloat16()
    for dil in (2, 4):
        o = nat.conv_gemm(a, w3, taps=9, bias=bias.repeat(2), act=2, dilation=dil)
        wf = w3.float().view(128, 9, 128).permute(0, 2, 1).reshape(128, 128, 3, 3)
        r = F.relu(F.conv2d(a.float().permute(0, 3, 1, 2), wf, bias.repeat(2), padding=dil, dilation=dil)).permute(0, 2, 3, 1)
        assert _rel(o, r) < 1e-2
    buf = torch.zeros(2, 28, 28, 384, dtype=torch.bfloat16, device=DEV)
    w1 = (torch.randn(256, 128, generator=g) / math.sqrt(128)).to(DEV).bfloat16()
    res = (torch.randn(2, 28, 28, 256, generator=g) * 0.5).to(DEV).bfloat16()
    nat.conv_gemm(a, w1, taps=1, res=res, res_mode=1, act=2, out=buf[..., 128:])
    torch.cuda.synchronize()
    r = F.relu(a.float() @ w1.float().t() + res.float())
    assert _rel(buf[..., 128:], r) < 1e-2 and buf[..., :128].abs().max().item() == 0
    # a channel slice as the A operand
    o2 = nat.conv_gemm(buf[..., 128:], (torch.randn(64, 256, generator=g) / 16).to(DEV).bfloat16(), taps=1)
    assert tuple(o2.shape) == (2, 28, 28, 64)


@pytest.mark.parametrize("B,C,H,W", [(8, 16, 64, 64), (5, 6, 48, 80)])
def test_batch_augment_matches_torchvision(B, C, H, W):
    """b200_augment against torchvision's own RandomAffine / flips applied per sample on the CPU with the same
    drawn parameters (code/prepare_single_model.py:107-113).  Index work: exact, except where a source coordinate
    lands within rounding of a pixel boundary (fp32 grid arithmetic in a different order) - at most 1e-4 of pixels."""
    import dataset as ds
    from torchvision.transforms import functional as TF
    from torchvision.transforms import InterpolationMode

    g = torch.Generator().manual_seed(B * 100 + H)
    x = torch.rand(B, C, H, W, generator=g)
    aug = ds.BatchAugment()
    torch.manual_seed(17)
    params = aug.sample_params(B, H, W)
    assert any(p[4] for p in params) or any(p[5] for p in params)
    got = aug.batch(x.to(DEV), params=params).cpu()
    bad = 0
    for b, (angle, tr, sc, sh, hf, vf) in enumerate(params):
        ref = TF.affine(x[b], angle, list(tr), sc, list(sh), interpolation=InterpolationMode.NEAREST, fill=[0.0] * C)
        if hf:
            ref = TF.hflip(ref)
        if vf:
            ref = TF.vflip(ref)
        bad += int((ref != got[b]).any(dim=0).sum())
    assert bad <= 1e-4 * B * H * W, f"{bad} of {B * H * W} pixels differ"
    # identity parameters copy the input; flips alone are exact
    ident = [(0.0, (0, 0), 1.0, (0.0, 0.0), False, False)] * B
    assert torch.equal(aug.batch(x.to(DEV), params=ident).cpu(), x)
    fl = [(0.0, (0, 0), 1.0, (0.0, 0.0), True, b % 2 == 0) for b in range(B)]
    out = aug.batch(x.to(DEV), params=fl).cpu()
    for b in range(B):
        want = torch.flip(x[b], dims=[2, 1] if b % 2 == 0 else [2])
        assert torch.equal(out[b], want)


def test_standalone_submodule_forwards_vs_oracle():
    """SEBlock, ReconHead, Projector, ClassificationHead, FeatureDownAlign, MaskHeadResize, MaskGuidedSpatialAttention,
    ResNetLiteBlock_withRecon, FusionReduce, GatingAttention, CrossAttentionBlock called on their own (reference
    model_module.py:25-43, :49-97, :100-125, :131-215, :220-316, :323-396, :745-818) against the oracle's functional
    restatements with the same seeded weights."""
    import torch.nn.functional as F

    import model_module as mm
    from oracle import model_oracle as mo
    from oracle import params as op

    g = torch.Generator().manual_seed(21)
    dev = "cuda"

    def seeded(mod):
        sd = op.seeded_state_dict(op.shapes_of(mod.state_dict()), seed=13)
        mod.load_state_dict(sd)
        return mod.to(dev).eval(), mo.SD(sd)

    def rel(a, b):
        return (a.float().cpu() - b).abs().max().item() / max(b.abs().max().item(), 1e-12)

    x = torch.randn(3, 128, 32, 32, generator=g).bfloat16().float()
    se, sd = seeded(mm.SEBlock(128))
    y, w = se(x.to(dev))
    ry, rw = mo.se_block(x, sd)
    assert rel(y, ry) <= 1e-2 and rel(w, rw) <= 1e-3
    rh, sd = seeded(mm.ReconHead(128))
    assert rel(rh(x.to(dev)), mo.recon_head(x, sd)) <= 2e-2
    pr, sd = seeded(mm.Projector(128, 64))
    assert rel(pr(x.to(dev)), mo.projector(x, sd)) <= 2e-2
    ch, sd = seeded(mm.ClassificationHead(128, 4))
    assert rel(ch(x.to(dev)), mo.classification_head(x, sd)) <= 5e-3
    fa, sd = seeded(mm.FeatureDownAlign(128, 256, downsample=False))
    assert rel(fa(x.to(dev)), mo.feature_down_align(x, sd)) <= 2e-2
    mh, sd = seeded(mm.MaskHeadResize(128))
    mlog = mh(x.to(dev))
    assert rel(mlog, mo.mask_head(x, sd)) <= 2e-2
    ma, sd = seeded(mm.MaskGuidedSpatialAttention(128, 1))
    mref = mo.mask_head(x, mo.SD(op.seeded_state_dict(op.shapes_of(mm.MaskHeadResize(128).state_dict()), seed=13)))
    ym, am = ma(x.to(dev), mref.to(dev))
    rym, ram = mo.mask_spatial_attention(x, mref, sd)
    assert rel(ym, rym) <= 1e-2 and rel(am, ram) <= 1e-3
    blk, sd = seeded(mm.ResNetLiteBlock_withRecon(128, 256, recon_ch=1, use_se=True, dropout=0.2))
    out, rec = blk(x.to(dev))
    rout, rrec = mo.res_block(x, sd, 1, 1, False, True)
    assert rel(out, rout) <= 2e-2 and rel(rec, rrec) <= 2e-2
    fr, sd = seeded(mm.FusionReduce(128, 64))
    assert rel(fr(x.to(dev)), F.gelu(mo._bn(mo._conv(x, sd.sub("reduce.0")), sd.sub("reduce.1")))) <= 2e-2
    # per-case vector blocks of the fusion head
    ga, sd = seeded(mm.GatingAttention(128, use_mask_attention=True))
    pd_, pc_ = torch.randn(5, 128, generator=g), torch.randn(5, 128, generator=g)
    md, mc = torch.randn(5, 1, 32, 32, generator=g), torch.randn(5, 1, 32, 32, generator=g)
    xin = torch.cat([pd_, pc_, md.mean(dim=(2, 3)), mc.mean(dim=(2, 3))], dim=1)
    ref = torch.softmax(F.linear(xin, sd["fc.weight"], sd["fc.bias"]), dim=1)
    assert rel(ga(pd_.to(dev), pc_.to(dev), md.to(dev), mc.to(dev)), ref) <= 1e-4
    ca = mm.CrossAttentionBlock(128, num_heads=4)
    ca.load_state_dict(op.seeded_state_dict(op.shapes_of(ca.state_dict()), seed=13))
    q, kv = torch.randn(5, 16, 128, generator=g), torch.randn(5, 16, 128, generator=g)
    with torch.no_grad():
        ao, aw = ca.cross_attn(q, kv, kv, need_weights=True)
        ref_out = ao + ca.attn_ffn(ao)
    ca.to(dev)
    got_out, got_w = ca(q.to(dev), kv.to(dev))
    assert rel(got_out, ref_out) <= 1e-4 and rel(got_w, aw) <= 1e-4


def test_paired_tiles_are_bitwise_the_unpaired_result():
    """conv_gemm_kernel<128, ..., PAIR> (two M tiles per CTA iteration sharing one weight slab, used once a launch has
    >= 2 x 148 M tiles) against the unpaired kernel on the same maps: the accumulation order per tile is the same, so the
    bf16 outputs must be bit-identical.  3x3 and 1x1, plain and residual + GELU epilogues, odd tile counts."""
    import b200_native as nat

    g = torch.Generator().manual_seed(8)
    for taps, cin, cout, res, hw in ((9, 128, 128, False, 32), (1, 128, 128, True, 32), (1, 512, 128, False, 32),
                                     (1, 128, 384, False, 32), (9, 128, 128, False, 14), (1, 256, 128, True, 14),
                                     (1, 64, 64, False, 32), (9, 64, 64, False, 32), (1, 128, 64, True, 32),
                                     (1, 256, 192, False, 32)):  # N = 64 tiles pair too
        # 32 x 32 maps: 41 cases x 8 tiles = 328 M tiles (>= 296: paired; odd pair count per N tile walk);
        # 14 x 14 maps (ragged 126-row tiles, two per case, direct epilogue): 163 cases = 326 M tiles
        B = 41 if hw == 32 else 163
        x = torch.randn(B, hw, hw, cin, generator=g).bfloat16().to(DEV)
        w = (torch.randn(cout, taps * cin, generator=g) / (taps * cin) ** 0.5).bfloat16().to(DEV)
        sc = (1 + 0.1 * torch.randn(cout, generator=g)).to(DEV)
        bi = (0.1 * torch.randn(cout, generator=g)).to(DEV)
        r = torch.randn(B, hw, hw, cout, generator=g).bfloat16().to(DEV) if res else None
        kw = dict(taps=taps, scale=sc, bias=bi, act=1, res=r, res_mode=1 if res else 0)
        big = nat.conv_gemm(x, w, **kw)
        for lo in (0, 17, 33):  # 8-case launches: 64 M tiles, below the pairing threshold
            kw_s = dict(kw, res=r[lo:lo + 8].contiguous() if res else None)
            small = nat.conv_gemm(x[lo:lo + 8].contiguous(), w, **kw_s)
            assert torch.equal(big[lo:lo + 8], small), (taps, cin, cout, res, hw, lo)
    # the tap-dot epilogue (3x3 128->128 + GELU + nine per-pixel dots, no map store: the reconstruction heads) pairs too
    B = 41
    x = torch.randn(B, 32, 32, 128, generator=g).bfloat16().to(DEV)
    w = (torch.randn(128, 9 * 128, generator=g) / (9 * 128) ** 0.5).bfloat16().to(DEV)
    sc, bi = (1 + 0.1 * torch.randn(128, generator=g)).to(DEV), (0.1 * torch.randn(128, generator=g)).to(DEV)
    dw = torch.randn(9, 128, generator=g).to(DEV)
    big = torch.full((B, 32, 32, 9), float("nan"), device=DEV)
    nat.conv_gemm(x, w, taps=9, scale=sc, bias=bi, act=1, store=False, dot_w=dw, dot_out=big, dot_bias=0.25)
    ref_map = nat.conv_gemm(x, w, taps=9, scale=sc, bias=bi, act=1).float()   # the stored (bf16-rounded) map
    ref = torch.einsum("bhwc,kc->bhwk", ref_map, dw) + 0.25
    assert (big - ref).abs().max().item() <= 2e-2 * ref.abs().max().item()     # dots of the un-rounded fp32 values
    for lo in (0, 17, 33):
        small = torch.empty((8, 32, 32, 9), device=DEV)
        nat.conv_gemm(x[lo:lo + 8].contiguous(), w, taps=9, scale=sc, bias=bi, act=1, store=False, dot_w=dw,
                      dot_out=small, dot_bias=0.25)
        assert torch.equal(big[lo:lo + 8], small), ("tap-dot", lo)


def test_reinitialised_weights_are_repacked():
    """forward -> initialize_model (in-place `.data` writes, version counters untouched) -> forward must use the new
    weights: the second result differs from the first and equals a fresh module holding the same state."""
    import model_module as mm
    import parameters_default as pd

    p = pd.default_parameters()
    torch.manual_seed(3)
    m = mm.ModelMaskHeadBackbone("dce", p).to(DEV).eval()
    x = torch.rand(2, 6, 64, 64, device=DEV)
    with torch.no_grad():
        a = m(x)[0].clone()
        mm.initialize_model(m, True)
        b = m(x)[0].clone()
        fresh = mm.ModelMaskHeadBackbone("dce", p)
        fresh.load_state_dict(m.state_dict())
        c = fresh.to(DEV).eval()(x)[0]
    # channel sums are float atomics: two runs agree to rounding, not bitwise
    assert not torch.allclose(a, b, rtol=1e-2, atol=1e-4) and torch.allclose(b, c, rtol=1e-3, atol=1e-5)


def test_standalone_transformer_forwards_vs_fp32_torch():
    """PatchEmbed, MultiHeadSelfAttention, MLP, TransformerBlock, TransformerEncoder and TransformerStage called on
    their own (transformer_model.py:7-175) against an fp32 torch evaluation of the same formulas with the same
    parameters (eval mode: the dropouts are identity)."""
    import transformer_model as tm

    def ref_attn(at, x):
        B, N, C = x.shape
        qkv = F.linear(x, at.qkv.weight, at.qkv.bias).reshape(B, N, 3, at.num_heads, at.head_dim).permute(2, 0, 3, 1, 4)
        a = (qkv[0] @ qkv[1].transpose(-2, -1) * at.scale).softmax(-1)
        return F.linear((a @ qkv[2]).transpose(1, 2).reshape(B, N, C), at.proj.weight, at.proj.bias)

    def ref_mlp(m, x):
        return F.linear(F.gelu(F.linear(x, m.fc1.weight, m.fc1.bias)), m.fc2.weight, m.fc2.bias)

    def ref_block(b, x):
        x = x + ref_attn(b.attn, F.layer_norm(x, (x.shape[-1],), b.norm1.weight, b.norm1.bias, b.norm1.eps)) * b.gamma1
        return x + ref_mlp(b.mlp, F.layer_norm(x, (x.shape[-1],), b.norm2.weight, b.norm2.bias, b.norm2.eps)) * b.gamma2

    def ref_stage(st, x):
        t = st.patch_embed.proj(x)
        hw = t.shape[-2:]
        t = t.flatten(2).transpose(1, 2)
        t = F.layer_norm(t, (t.shape[-1],), st.patch_embed.norm.weight, st.patch_embed.norm.bias, st.patch_embed.norm.eps)
        for b in st.transformer.layers:
            t = ref_block(b, t)
        return t.transpose(1, 2).reshape(x.shape[0], -1, *hw)

    torch.manual_seed(5)
    stage = tm.TransformerStage(in_ch=256, embed_dim=512, depth=2, heads=4).to(DEV).eval()
    with torch.no_grad():
        for p_ in stage.parameters():  # non-trivial LayerNorm / LayerScale parameters
            if p_.dim() == 1:
                p_.add_(0.2 * torch.randn_like(p_))
        x = torch.randn(3, 256, 16, 16, device=DEV)          # -> 64 tokens
        tok = torch.randn(3, 64, 512, device=DEV)
        blk = stage.transformer.layers[0]
        tokens, hw = stage.patch_embed(x)
        assert tuple(tokens.shape) == (3, 64, 512) and tuple(hw) == (8, 8) and tokens.dtype == torch.float32
        cases = {"attn": (blk.attn(tok), ref_attn(blk.attn, tok)), "mlp": (blk.mlp(tok), ref_mlp(blk.mlp, tok)),
                 "block": (blk(tok), ref_block(blk, tok)),
                 "encoder": (stage.transformer(tok), ref_block(stage.transformer.layers[1], ref_block(blk, tok))),
                 "stage": (stage(x), ref_stage(stage, x))}
        torch.cuda.synchronize()
        for name, (got, ref) in cases.items():
            assert got.shape == ref.shape and got.dtype == torch.float32, name
            assert _rel(got, ref) < 1.5e-2, (name, _rel(got, ref))
        stage.train()
        with pytest.raises(NotImplementedError):
            stage(x)


@pytest.mark.parametrize("B,H,W,Cin,Cout,taps,res_mode", [(20, 14, 14, 128, 256, 9, 0), (9, 14, 14, 64, 128, 1, 1),
                                                         (5, 7, 7, 128, 64, 9, 2), (37, 14, 14, 192, 768, 9, 0),
                                                         (163, 14, 14, 128, 128, 9, 1)])
def test_conv_gemm_tiles_spanning_cases(B, H, W, Cin, Cout, taps, res_mode):
    """Small ragged maps are tiled across cases (14 x 14: one image row of 9 consecutive cases per 128-row tile, 126 rows
    filled, instead of 9-row tiles of one case): same results as a per-case launch (which cannot span cases) bit for
    bit, and as fp32 torch within bf16 rounding; batch sizes that leave a partial last group, and the paired kernel."""
    g = torch.Generator().manual_seed(B + H)
    x = torch.randn(B, H, W, Cin, generator=g).bfloat16().to(DEV)
    w = (torch.randn(Cout, taps * Cin, generator=g) / (taps * Cin) ** 0.5).bfloat16().to(DEV)
    sc = (1 + 0.1 * torch.randn(Cout, generator=g)).to(DEV)
    bi = (0.1 * torch.randn(Cout, generator=g)).to(DEV)
    r = torch.randn(B, H, W, Cout, generator=g).bfloat16().to(DEV) if res_mode else None
    y = nat.conv_gemm(x, w, taps=taps, scale=sc, bias=bi, act=1, res=r, res_mode=res_mode)
    for b in (0, B // 2, B - 1):
        one = nat.conv_gemm(x[b:b + 1].contiguous(), w, taps=taps, scale=sc, bias=bi, act=1,
                            res=None if r is None else r[b:b + 1].contiguous(), res_mode=res_mode)
        assert torch.equal(y[b:b + 1], one), (b,)
    k = int(taps ** 0.5)
    wt = w.float().view(Cout, k, k, Cin).permute(0, 3, 1, 2)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wt, padding=k // 2) * sc.view(1, -1, 1, 1) + bi.view(1, -1, 1, 1)
    if res_mode == 1:
        ref = F.gelu(ref + r.float().permute(0, 3, 1, 2))
    else:
        ref = F.gelu(ref)
        if res_mode == 2:
            ref = ref + r.float().permute(0, 3, 1, 2)
    assert _rel(y.permute(0, 3, 1, 2), ref) < 1.5e-2


@pytest.mark.parametrize("B,H,W,C", [(5, 32, 32, 128), (3, 32, 32, 512), (4, 14, 14, 768), (2, 7, 9, 24), (3, 16, 16, 256)])
def test_scale_map_channel_gate_and_pixel_attention(B, H, W, C):
    """y = x * gate[b, c] * (1 + gamma * attn[b, p]) (SE rescale model_module.py:43, mask-guided modulation :96): both index
    paths of the kernel (C / 8 a power of two dividing the block: shared gate registers and shifts; any other C), each
    factor alone and together, against fp32 torch."""
    g = torch.Generator().manual_seed(C + B)
    x = torch.randn(B, H, W, C, generator=g).bfloat16().to(DEV)
    gate = torch.rand(B, C, generator=g).to(DEV)
    attn = torch.rand(B, H * W, generator=g).to(DEV)
    gamma = torch.tensor([0.7], device=DEV)
    xf = x.float()
    cases = {"gate": (gate, None, None, xf * gate.view(B, 1, 1, C)),
             "attn": (None, attn, gamma, xf * (1 + 0.7 * attn.view(B, H, W, 1))),
             "both": (gate, attn, gamma, xf * gate.view(B, 1, 1, C) * (1 + 0.7 * attn.view(B, H, W, 1)))}
    for name, (ga, at, gm, ref) in cases.items():
        y = nat.scale_map(x, torch.empty_like(x), gate=ga, attn=at, gamma=gm)
        torch.cuda.synchronize()
        assert _rel(y, ref) < 6e-3, (name, _rel(y, ref))
