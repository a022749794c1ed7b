"""Attention over more than 256 tokens: the key-tiled fused attention kernel behind b200_attention /
b200_attention_mc (attn_long_kernel), against fp32 torch, its rescale paths, its dropout rule bit for bit, and the
transformers that use it (ViT-B/16 at 256 x 256, the hybrid stage at 128 x 128 ROIs) against the oracle."""
import math

import numpy as np
import pytest
import torch

import b200_native as nat

pytestmark = pytest.mark.gpu
DEV = "cuda"
P = 0.1
TAU = 8.0  # log2 units: a key tile moves the row's reference only when its max exceeds it by more than this


def _rel(got, ref):
    return (got.float() - ref.float()).abs().max().item() / ref.float().abs().max().item()


def _within_binomial(dropped, n, p, sigmas=5.0):
    return abs(dropped / n - p) <= sigmas * math.sqrt(p * (1 - p) / n)


def _split(qkv, B, N, heads, dh):
    return (qkv.float().view(B, N, 3, heads, dh).permute(2, 0, 3, 1, 4)[i] for i in range(3))


def _reference(qkv, B, N, heads, dh):
    q, k, v = _split(qkv, B, N, heads, dh)
    return (torch.softmax(q @ k.transpose(-1, -2) * dh ** -0.5, dim=-1) @ v).permute(0, 2, 1, 3).reshape(B * N, -1)


def _buffers(x, B, N, heads, dh, pad):
    """x [B*N, 3C] -> bf16 qkv view in a NaN-padded buffer, and an output view whose padding holds NaN sentinels."""
    C = heads * dh
    buf = torch.full((B * N, 3 * C + pad), float("nan"), dtype=torch.bfloat16, device=DEV)
    qkv = buf[:, :3 * C]
    qkv.copy_(x.bfloat16())
    out_buf = torch.full((B * N, C + pad), float("nan"), dtype=torch.bfloat16, device=DEV)
    return qkv, out_buf, out_buf[:, :C]


@pytest.mark.parametrize("B,heads,N,dh,pad", [
    (2, 4, 257, 128, 0), (2, 4, 384, 128, 0), (2, 2, 1000, 128, 0), (1, 4, 1024, 128, 0), (1, 2, 4096, 128, 0),
    (2, 4, 257, 64, 0), (2, 4, 384, 64, 0), (2, 2, 1000, 64, 0), (1, 4, 1024, 64, 0), (1, 2, 4096, 64, 0),
    (4, 12, 257, 64, 0),       # ViT-B/16 at 256 x 256: 16 x 16 patches + cls
    (3, 2, 1000, 128, 24),     # ragged N, padded qkv_ld / out_ld
    (2, 4, 1000, 64, 8),
    (40, 12, 257, 64, 0),      # 1440 work items: more than resident CTAs (persistent loop)
    (1, 1, 16384, 128, 0),     # the documented limit: a 128 x 128 token grid
])
def test_long_attention_vs_fp32(B, heads, N, dh, pad):
    g = torch.Generator(device="cpu").manual_seed(B * heads + N + dh)
    C = heads * dh
    qkv, out_buf, out = _buffers(torch.randn(B * N, 3 * C, generator=g) * 0.9, B, N, heads, dh, pad)
    nat.attention(qkv, out, B, N, heads, dh)
    torch.cuda.synchronize()
    ref = _reference(qkv, B, N, heads, dh)
    assert torch.isfinite(out.float()).all()
    err = _rel(out, ref)
    print(f"attention ({B},{heads},{N},{dh}) pad {pad}: max|d|/max|ref| = {err:.2e}")
    assert err < 1.2e-2
    if pad:
        assert torch.isnan(out_buf[:, C:].float()).all()  # padding columns untouched


# ------------------------------------------------------------------ rescale paths ----
RB, RH, RN, RD = 2, 3, 1025, 64  # 9 key tiles, the last one holds the single key 1024


def _rescale_input(seed=31):
    """Three heads, one situation each:
    head 0: K rows of the first key tile scaled up -> every row's max sits in tile 0, the reference never moves;
    head 1: q and k share a direction w and K grows with the key index -> every tile's max exceeds the previous one
            by ~16 (log2 units) > TAU, so every full tile after the first rescales;
    head 2: the last key (alone in the ragged last tile) is aligned with every query -> it holds the row max and
            moves the reference in the last tile."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    C = RH * RD
    x = torch.randn(RB, RN, 3, RH, RD, generator=g) * 0.5
    x[:, :128, 1, 0] *= 4.0
    w = torch.ones(RD)
    a = torch.arange(RN, dtype=torch.float32) / 128.0 * 1.4
    x[:, :, 0, 1] = 0.3 * x[:, :, 0, 1] + w
    x[:, :, 1, 1] = 0.3 * x[:, :, 1, 1] + a[None, :, None] * w
    x[:, :, 0, 2] = x[:, :, 0, 2] + 0.5 * w
    x[:, RN - 1, 1, 2] = 3.0 * w
    return x.reshape(RB * RN, 3 * C)


def _reference_moves(qkv):
    """The kernel's reference rule replayed on the fp32 scores: per (case, head, row), the key tiles that move it, and
    the key of the row max."""
    q, k, _ = _split(qkv, RB, RN, RH, RD)
    s = (q @ k.transpose(-1, -2)) * RD ** -0.5 * math.log2(math.e)
    nt = (RN + 127) // 128
    tmax = torch.stack([s[..., 128 * j:128 * (j + 1)].amax(-1) for j in range(nt)], -1)  # [B, H, N, tiles]
    m = tmax[..., 0].clone()
    moves = torch.zeros_like(tmax, dtype=torch.bool)
    for j in range(1, nt):
        moves[..., j] = tmax[..., j] > m + TAU
        m = torch.where(moves[..., j], tmax[..., j], m)
    return moves, s.argmax(-1)


def test_long_attention_rescale_paths():
    qkv, _, out = _buffers(_rescale_input(), RB, RN, RH, RD, 0)
    moves, argmax = _reference_moves(qkv)
    # each situation really occurs in the input
    assert (argmax[:, 0] < 128).all() and not moves[:, 0].any()         # head 0: max in tile 0, never rescales
    assert moves[:, 1, :, 1:-1].all()                                   # head 1: every later full tile rescales
    assert (argmax[:, 2] == RN - 1).all() and moves[:, 2, :, -1].all()  # head 2: the single last key moves it
    nat.attention(qkv, out, RB, RN, RH, RD)
    torch.cuda.synchronize()
    ref = _reference(qkv, RB, RN, RH, RD)
    assert torch.isfinite(out.float()).all()
    for h in range(RH):
        sl = slice(h * RD, (h + 1) * RD)
        err = _rel(out[:, sl], ref[:, sl])
        print(f"rescale input, head {h}: max|d|/max|ref| = {err:.2e}")
        assert err < 1.2e-2, h


# ------------------------------------------------------------------------ dropout ----
def _attention_probs(qkv, B, N, heads, dh, pad, dropout):
    """Reads the (dropped, rescaled) probabilities off the kernel's output: with V one-hot on keys [j0, j0 + dh),
    O[q, d] = P'[q, j0 + d].  ceil(N / dh) launches with the same dropout (p, seed) -> P' [B, heads, N, N] fp32."""
    C = heads * dh
    out_buf = torch.zeros(B * N, C + pad, dtype=torch.bfloat16, device=DEV)
    out = out_buf[:, :C]
    pp = torch.empty(B, heads, N, N, device=DEV)
    eye = torch.eye(dh, dtype=torch.bfloat16, device=DEV)
    for j0 in range(0, N, dh):
        v = torch.zeros(N, dh, dtype=torch.bfloat16, device=DEV)
        w = min(dh, N - j0)
        v[j0:j0 + w] = eye[:w]
        qkv[:, 2 * C:].copy_(v.view(1, N, 1, dh).expand(B, N, heads, dh).reshape(B * N, C))
        nat.attention(qkv, out, B, N, heads, dh, dropout=dropout)
        o = out.float().view(B, N, heads, dh).permute(0, 2, 1, 3)  # [B, heads, q, d]
        pp[..., j0:j0 + w] = o[..., :w]
        if pad:
            assert torch.count_nonzero(out_buf[:, C:]) == 0
    torch.cuda.synchronize()
    return pp


def _qkv(B, N, heads, dh, pad, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    C = heads * dh
    buf = torch.zeros(B * N, 3 * C + pad, dtype=torch.bfloat16, device=DEV)
    qkv = buf[:, :3 * C]
    qkv.copy_((torch.randn(B * N, 3 * C, generator=g) * 0.9).bfloat16())
    return qkv


def _philox4x32_7(ctr, seed):
    """Philox4x32-7 of 64-bit counters (numpy uint64 array) under a 64-bit key -> [4, n] uint32 words."""
    M32 = np.uint64(0xFFFFFFFF)
    c0, c1 = ctr & M32, ctr >> np.uint64(32)
    c2 = np.full_like(c0, 0x2545F491)
    c3 = np.full_like(c0, 0x9E3779B9)
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)
    for _ in range(7):
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & M32
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & M32, (k1 + np.uint64(0xBB67AE85)) & M32
    return np.stack([c0, c1, c2, c3])


def _documented_mask(B, N, heads, p, seed):
    """The dropout rule of b200_attention_mc: (b, h, n, j) is dropped when word j % 4 of
    Philox4x32-7(seed; ((b * heads + h) * N + n) * 64 * ceil(N / 256) + j / 4) < p * 2^32."""
    rows = np.arange(B * heads * N, dtype=np.uint64) * np.uint64(64 * ((N + 255) // 256))
    ctr = (rows[:, None] + np.arange((N + 3) // 4, dtype=np.uint64)[None, :]).reshape(-1)
    words = _philox4x32_7(ctr, seed).reshape(4, B * heads * N, -1).transpose(1, 2, 0).reshape(B * heads * N, -1)[:, :N]
    thresh = min(int(float(np.float32(p)) * 4294967296.0), 0xFFFFFFFF)
    return torch.from_numpy(words < thresh).view(B, heads, N, N)


@pytest.mark.parametrize("B,heads,N,dh,pad", [(2, 3, 257, 64, 8), (1, 2, 1024, 128, 0), (1, 2, 1000, 64, 0)])
def test_long_attention_dropout_mask_read_off_the_output(B, heads, N, dh, pad):
    qkv = _qkv(B, N, heads, dh, pad, seed=B * heads + N)
    q, k, _ = _split(qkv, B, N, heads, dh)
    ref = torch.softmax(q @ k.transpose(-1, -2) * dh ** -0.5, dim=-1) / (1 - P)
    got = _attention_probs(qkv, B, N, heads, dh, pad, (P, 1234))
    dropped = got == 0
    assert not (ref == 0).any()  # every probability is readable (none underflows)
    kept_err = ((got - ref).abs() / ref)[~dropped].max().item()
    n = dropped.numel()
    print(f"attention ({B},{heads},{N},{dh}) p={P}: drop rate {dropped.sum().item() / n:.5f} over {n} probabilities, "
          f"worst kept relative error {kept_err:.2e}")
    assert kept_err < 1e-2
    assert _within_binomial(dropped.sum().item(), n, P)
    # per head, per 128-query tile, per 128-key tile
    for dim, size in ((1, 1), (2, 128), (3, 128)):
        for s0 in range(0, dropped.shape[dim], size):
            part = dropped.narrow(dim, s0, min(size, dropped.shape[dim] - s0))
            assert _within_binomial(part.sum().item(), part.numel(), P), (dim, s0)
    # bit for bit the documented rule
    assert torch.equal(dropped.cpu(), _documented_mask(B, N, heads, P, 1234))
    # the same seed gives the same mask, another seed another one
    again = _attention_probs(qkv, B, N, heads, dh, pad, (P, 1234))
    assert torch.equal(again, got)
    other = _attention_probs(qkv, B, N, heads, dh, pad, (P, 1235)) == 0
    assert (other != dropped).float().mean().item() > 0.5 * 2 * P * (1 - P)


def test_long_attention_dropout_mask_depends_on_indices_only():
    """The random input and the rescale input (every tile moving the reference in head 1) give the same mask."""
    C = RH * RD
    masks = []
    for x in (torch.randn(RB * RN, 3 * C, generator=torch.Generator().manual_seed(4)) * 0.9, _rescale_input()):
        qkv, _, _ = _buffers(x, RB, RN, RH, RD, 0)
        full = _attention_probs(qkv, RB, RN, RH, RD, 0, (0.0, 0))
        got = _attention_probs(qkv, RB, RN, RH, RD, 0, (P, 99))
        readable = full > 1e-30  # steep rows underflow to zeros or bf16 subnormals, which cannot show a 1 / (1 - p)
        kept = readable & (got != 0)
        ratio = (got[kept] / full[kept] * (1 - P) - 1).abs().max().item()
        print(f"{readable.float().mean().item():.3f} of the probabilities readable, kept / undropped ratio off "
              f"1 / (1 - p) by at most {ratio:.2e}")
        assert ratio < 1e-2
        masks.append((got == 0, readable))
    both = masks[0][1] & masks[1][1]
    assert both.sum().item() > 0.3 * both.numel()
    assert torch.equal(masks[0][0][both], masks[1][0][both])
    assert torch.equal(masks[1][0][masks[1][1]].cpu(), _documented_mask(RB, RN, RH, P, 99)[masks[1][1].cpu()])


def test_long_attention_dropout_p0_is_the_plain_kernel_and_mean_is_unbiased():
    B, heads, N, dh = 1, 2, 1024, 128
    qkv = _qkv(B, N, heads, dh, 0, seed=5)
    C = heads * dh
    o0 = torch.empty(B * N, C, dtype=torch.bfloat16, device=DEV)
    nat.attention(qkv, o0, B, N, heads, dh)
    oz = torch.empty_like(o0)
    nat.attention(qkv, oz, B, N, heads, dh, dropout=(0.0, 7))
    torch.cuda.synchronize()
    assert torch.equal(o0, oz)
    outs = torch.empty(64, B * N, C)
    o = torch.empty_like(o0)
    for i in range(64):
        nat.attention(qkv, o, B, N, heads, dh, dropout=(P, 1000 + i))
        outs[i] = o.float().cpu()
    mean, se = outs.mean(0), outs.std(0) / 8.0
    rms = lambda t: t.pow(2).mean().sqrt().item()
    err, mc, ref = rms(mean - o0.float().cpu()), rms(se), rms(o0.float().cpu())
    print(f"attention mean of 64 dropout passes vs undropped: rms error {err:.3e}, rms Monte-Carlo error {mc:.3e}")
    assert err <= 1.3 * mc + 4e-3 * ref
    assert mc > 0


# -------------------------------------------------------------------- model level ----
MODEL_TOL = 2e-2
VIT_TOL = 6e-2     # maps downstream of the ViT path's first GroupNorm backbone mix (tests/test_parity_gpu.py VIT_TOL)
VIT_UPSTREAM = ("aux.raw_feats.0", "aux.recon_feats.0", "aux.proj_pairs.0", "aux.proj_pairs.1", "aux.mod_attn_map")
# At 256 x 256 the fp32 oracle with nothing but its GEMM operands rounded to bf16 (tests/tools/bf16_floor_vit256.py)
# already deviates from itself by 1.3-2.1 % on the maps upstream of the first backbone mix (224 x 224: 1.2-1.7 %), so
# those are held to 3e-2 here instead of 2e-2 (DESIGN.md section 2).
VIT256_UPSTREAM_TOL = 3e-2
HYBRID_FUSED_TOL = 3e-2  # fused outputs of the hybrid configuration (tests/test_parity_gpu.py)


def _relmax(got, ref):
    got, ref = got.detach().float().cpu(), ref.detach().float().cpu()
    return (got - ref).abs().max().item() / max(ref.abs().max().item(), 1e-12)


def _inputs(n, size, seed):
    from oracle import params as op

    dwi_raw, dce_raw, _, _ = op.synthetic_raw(n, seed=seed, size=size, kind="S")
    return dwi_raw / dwi_raw.amax(dim=(1, 2, 3), keepdim=True), dce_raw


def _modules(p, seed, backbones=None):
    """Product encoders + fusion head with seeded weights, and the state dicts the oracle reads."""
    import model_module as mm
    from oracle import params as op

    backbones = backbones or {}
    mods = {"dwi": mm.ModelMaskHeadBackbone("dwi", p, backbones.get("dwi")),
            "dce": mm.ModelMaskHeadBackbone("dce", p, backbones.get("dce")), "fusion": mm.FusionModel(p)}
    sds = {}
    for k, m in mods.items():
        sds[k] = op.seeded_state_dict(op.shapes_of(m.state_dict()), seed=seed)
        m.load_state_dict(sds[k])
        m.to(DEV).eval()
    return sds, mods


def _product_and_oracle(p, sds, mods, dwi, dce):
    from oracle import model_oracle as mo

    with torch.no_grad():
        ld, ad, md = mods["dwi"](dwi.to(DEV))
        lc, ac, mc = mods["dce"](dce.to(DEV))
        lf, mf, af = mods["fusion"](ad["raw_feats"], ac["raw_feats"], md, mc)
    torch.cuda.synchronize()
    torch.set_num_threads(max(torch.get_num_threads(), 8))
    with torch.no_grad():
        o_d = mo.encoder_forward(sds["dwi"], "dwi", p, dwi)
        o_c = mo.encoder_forward(sds["dce"], "dce", p, dce)
        o_f = mo.fusion_forward(sds["fusion"], p, o_d[1]["raw_feats"], o_c[1]["raw_feats"], o_d[2], o_c[2])
    got = {"dwi/logits": ld, "dwi/aux": ad, "dwi/mask": md, "dce/logits": lc, "dce/aux": ac, "dce/mask": mc,
           "fusion/logits": lf, "fusion/mask": mf, "fusion/aux": af}
    ref = {"dwi/logits": o_d[0], "dwi/aux": o_d[1], "dwi/mask": o_d[2], "dce/logits": o_c[0], "dce/aux": o_c[1],
           "dce/mask": o_c[2], "fusion/logits": o_f[0], "fusion/mask": o_f[1], "fusion/aux": o_f[2]}
    import golden_util as gu

    errs = {}
    for prefix in got:
        for (k, a), (_, b) in zip(gu.walk(prefix, got[prefix]), gu.walk(prefix, ref[prefix])):
            assert tuple(a.shape) == tuple(b.shape), k
            errs[k] = _relmax(a, b)
    return errs, got


def _vit_parameters(size):
    import foundation_model as fm
    import parameters_default as pd

    p = pd.default_parameters(input_size=size)
    backbones = {}
    for m, c in (("dwi", 16), ("dce", 6)):
        mp = p[f"{m}_model_parameters"]
        mp["backbone_str"], mp["use_backbone"] = "vit_base_patch16_224", True
        backbones[m] = fm.build_medical_backbone(p, None, m, in_channels=c)
    fs = p["fusion_model_parameters"]["fusion_specific_parameters"]
    fs["dwi_out_channels"] = fs["dce_out_channels"] = 768
    return p, backbones


def test_vit_backbone_at_256_vs_oracle():
    """ViT-B/16 at the reference's default input size 256: 257 tokens, all 12 feature maps [B, 768, 16, 16]."""
    import foundation_model as fm
    import parameters_default as pd
    from oracle import backbone_oracle as bo
    from oracle import params as op

    p = pd.default_parameters(input_size=256)
    p["dce_model_parameters"]["backbone_str"] = "vit_base_patch16_224"
    p["dce_model_parameters"]["use_backbone"] = True
    bb = fm.build_medical_backbone(p, torch.device(DEV), "dce", in_channels=6)
    shapes = {k: tuple(v.shape) for k, v in bb.state_dict().items()}
    assert shapes == bo.vit_shapes(in_chans=6, img=256)
    sd = op.seeded_state_dict(shapes, seed=5)
    bb.load_state_dict(sd)
    x = torch.rand(2, 6, 256, 256, generator=torch.Generator().manual_seed(2))
    feats = bb(x.to(DEV))
    torch.cuda.synchronize()
    torch.set_num_threads(max(torch.get_num_threads(), 8))
    with torch.no_grad():
        ref = bo.vit_features(sd, x)
    assert len(feats) == 12 and tuple(feats[0].shape) == (2, 768, 16, 16)
    errs = [_relmax(a, b) for a, b in zip(feats, ref)]
    print("ViT at 256 x 256, feature errors per block:", [f"{e:.1e}" for e in errs])
    assert max(errs) <= MODEL_TOL


def test_vit_adapter_pipeline_at_256_vs_oracle():
    """use_backbone ViT encoders (BackboneAdapter necks, GroupNorm backbone mixes, heads on 16 x 16 maps) and the
    fusion head at input_size=256, against the oracle: 3e-2 upstream of the first backbone mix (the bf16 floor of this
    configuration is 2.1 % there), 6e-2 downstream."""
    p, backbones = _vit_parameters(256)
    sds, mods = _modules(p, 11, backbones)
    dwi, dce = _inputs(2, 256, 4321)
    errs, got = _product_and_oracle(p, sds, mods, dwi, dce)
    print("ViT path at 256 x 256, max|d|/max|ref|:", sorted(((k, f"{v:.1e}") for k, v in errs.items()),
                                                             key=lambda kv: -float(kv[1])))
    assert tuple(got["dwi/aux"]["raw_feats"][2].shape) == (2, 768, 16, 16) and got["fusion/logits"].shape == (2, 4)
    bad = {k: v for k, v in errs.items() if v > (VIT256_UPSTREAM_TOL if k.endswith(VIT_UPSTREAM) else VIT_TOL)}
    assert not bad, bad


def _hybrid128():
    import parameters_default as pd

    p = pd.default_parameters(input_size=128)
    for m in ("dwi", "dce"):
        p[f"{m}_model_parameters"]["use_hybrid_transformer"] = True
    return p


def test_hybrid_encoders_at_128_vs_oracle():
    """use_hybrid_transformer=True on 128 x 128 ROIs: the TransformerStage sees 32 x 32 = 1024 tokens."""
    p = _hybrid128()
    sds, mods = _modules(p, 7)
    dwi, dce = _inputs(2, 128, 1234)
    errs, got = _product_and_oracle(p, sds, mods, dwi, dce)
    print("hybrid at 128 x 128, max|d|/max|ref|:", sorted(((k, f"{v:.1e}") for k, v in errs.items()),
                                                          key=lambda kv: -float(kv[1])))
    assert tuple(got["dwi/aux"]["raw_feats"][2].shape) == (2, 512, 32, 32) and got["fusion/logits"].shape == (2, 4)
    bad = {k: v for k, v in errs.items() if v > (HYBRID_FUSED_TOL if k.startswith("fusion") else MODEL_TOL)}
    assert not bad, bad


@pytest.mark.parametrize("grid", [32, 64])
def test_standalone_transformer_stage_on_large_grids_vs_fp32_torch(grid):
    """transformer_model.TransformerStage on its own over a grid x grid token map (1024 / 4096 tokens)."""
    import torch.nn.functional as F

    import transformer_model as tm

    def ref_stage(st, x):
        t = st.patch_embed.proj(x)
        hw = t.shape[-2:]
        t = t.flatten(2).transpose(1, 2)
        t = F.layer_norm(t, (t.shape[-1],), st.patch_embed.norm.weight, st.patch_embed.norm.bias, st.patch_embed.norm.eps)
        for b in st.transformer.layers:
            at = b.attn
            h = F.layer_norm(t, (t.shape[-1],), b.norm1.weight, b.norm1.bias, b.norm1.eps)
            B, N, C = h.shape
            qkv = F.linear(h, at.qkv.weight, at.qkv.bias).reshape(B, N, 3, at.num_heads, at.head_dim).permute(2, 0, 3, 1, 4)
            a = (qkv[0] @ qkv[1].transpose(-2, -1) * at.scale).softmax(-1)
            t = t + F.linear((a @ qkv[2]).transpose(1, 2).reshape(B, N, C), at.proj.weight, at.proj.bias) * b.gamma1
            h = F.layer_norm(t, (t.shape[-1],), b.norm2.weight, b.norm2.bias, b.norm2.eps)
            t = t + F.linear(F.gelu(F.linear(h, b.mlp.fc1.weight, b.mlp.fc1.bias)), b.mlp.fc2.weight, b.mlp.fc2.bias) * b.gamma2
        return t.transpose(1, 2).reshape(x.shape[0], -1, *hw)

    torch.manual_seed(5)
    stage = tm.TransformerStage(in_ch=256, embed_dim=512, depth=2, heads=4).to(DEV).eval()
    with torch.no_grad():
        for p_ in stage.parameters():  # non-trivial LayerNorm / LayerScale parameters
            if p_.dim() == 1:
                p_.add_(0.2 * torch.randn_like(p_))
        x = torch.randn(2, 256, 2 * grid, 2 * grid, device=DEV)
        got, ref = stage(x), ref_stage(stage, x)
    torch.cuda.synchronize()
    assert got.shape == ref.shape == (2, 512, grid, grid) and got.dtype == torch.float32
    err = _relmax(got, ref)
    print(f"TransformerStage on {grid} x {grid} tokens: max|d|/max|ref| = {err:.2e}")
    assert err < 1.5e-2


def test_hybrid_mc_dropout_at_128_is_statistically_the_reference():
    """predict_mc_dropout with the hybrid encoders on 128 x 128 ROIs (attention dropout through the key-tiled kernel)
    against the MC-dropout oracle, and predict_tta_mc at the same size."""
    import mc_dropout_oracle as mdo
    import train_fusion as b_tf
    from oracle import model_oracle as mo

    p = _hybrid128()
    sds, mods = _modules(p, 7)
    lm = b_tf.LightningFusionModel(mods["dwi"], mods["dce"], mods["fusion"], p)
    n, passes = 2, 24
    dwi, dce = _inputs(n, 128, 22)
    lm.set_mc_seed(5)
    mean_a, std_a, _ = lm.predict_mc_dropout(dwi.to(DEV), dce.to(DEV), passes=passes)
    torch.cuda.synchronize()
    assert std_a.max().item() > 1e-4
    torch.manual_seed(3)
    torch.set_num_threads(max(torch.get_num_threads(), 8))
    ref = []
    with torch.no_grad():
        for _ in range(passes):
            _, ad, md = mdo.encoder_forward(sds["dwi"], "dwi", p, dwi, mc_dropout=True)
            _, ac, mc = mdo.encoder_forward(sds["dce"], "dce", p, dce, mc_dropout=True)
            ref.append(torch.softmax(mo.fusion_forward(sds["fusion"], p, ad["raw_feats"], ac["raw_feats"], md, mc)[0], 1))
    ref = torch.stack(ref)
    ref_mean, ref_std = ref.mean(0), ref.std(0)
    se = torch.sqrt(ref_std ** 2 + std_a.cpu() ** 2) / passes ** 0.5
    diff = (mean_a.cpu() - ref_mean).abs()
    ratio = (std_a.cpu().mean() / ref_std.mean()).item()
    print(f"hybrid MC dropout at 128 x 128: max |mean - oracle mean| {diff.max().item():.3e}, spread ratio {ratio:.3f}")
    assert (diff <= 5 * se + HYBRID_FUSED_TOL * ref_mean.max()).all(), (diff, se)
    assert 0.5 < ratio < 1.8, ratio
    mean_t, _, _ = lm.predict_tta_mc(dwi.to(DEV), dce.to(DEV), passes=2)
    assert mean_t.shape == (n, 4) and torch.isfinite(mean_t).all() and abs(mean_t.sum(1).mean().item() - 1) < 1e-3
