"""MC-dropout inference through the hybrid transformer stage: the attention dropout inside the fused attention kernel
(b200_attention_mc), the dropout before the residual in the fp32 epilogue of the tcgen05 GEMM (b200_linear_mc), and
the encoders' MC-dropout predictions against the oracle with the reference's per-module switches."""
import math

import pytest
import torch

import b200_native as nat
import mc_dropout_oracle as mdo
from oracle import model_oracle as mo
from oracle import params as op
from test_parity_gpu import _build, _lightning, _relmax, _run_product

pytestmark = pytest.mark.gpu
DEV = "cuda"
P = 0.1
HYBRID_TOL = 3e-2  # deterministic tolerance of the hybrid configuration's fused outputs (DESIGN.md section 2)


def _within_binomial(dropped, n, p, sigmas=5.0):
    return abs(dropped / n - p) <= sigmas * math.sqrt(p * (1 - p) / n)


# ------------------------------------------------------------------ attention ----
def _qkv(B, N, heads, dh, pad, seed, steep=False):
    g = torch.Generator(device="cpu").manual_seed(seed)
    C = heads * dh
    x = torch.randn(B * N, 3 * C, generator=g)
    if steep:  # the input of test_fused_attention_steep_rows_take_the_two_pass_path: cases 0-1 near one-hot rows
        x[: 2 * N, : 2 * C] *= 6.0
        x[2 * N:] *= 0.9
    else:
        x *= 0.9
    buf = torch.zeros(B * N, 3 * C + pad, dtype=torch.bfloat16, device=DEV)
    qkv = buf[:, :3 * C]
    qkv.copy_(x.bfloat16())
    return qkv


def _probs(qkv, B, N, heads, dh):
    """fp32 softmax of the bf16 q, k: [B, heads, N, N]."""
    q, k = (qkv.float().view(B, N, 3, heads, dh).permute(2, 0, 3, 1, 4)[i] for i in range(2))
    return torch.softmax(q @ k.transpose(-1, -2) * dh ** -0.5, dim=-1)


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


@pytest.mark.parametrize("B,heads,N,dh,pad", [(2, 4, 256, 128, 0), (3, 12, 197, 64, 0), (2, 2, 70, 64, 64),
                                              (40, 12, 197, 64, 0)])
def test_attention_dropout_mask_read_off_the_output(B, heads, N, dh, pad):
    qkv = _qkv(B, N, heads, dh, pad, seed=B * heads + N)
    ref = _probs(qkv, B, N, heads, dh) / (1 - P)
    got = _attention_probs(qkv, B, N, heads, dh, pad, (P, 1234))
    dropped = got == 0
    assert not (ref == 0).any()  # every probability is readable (none underflows)
    kept_err = ((got - ref).abs() / ref)[~dropped].max().item()
    n = dropped.numel()
    rate = dropped.sum().item() / n
    print(f"attention ({B},{heads},{N},{dh}) p={P}: drop rate {rate:.5f} over {n} probabilities, "
          f"worst kept relative error {kept_err:.2e}")
    assert kept_err < 1e-2
    assert _within_binomial(dropped.sum().item(), n, P)
    # per head, per 128-query tile, per 32-key chunk: the counter must not depend on the tiling
    for dim, size in ((1, 1), (2, 128), (3, 32)):
        for s0 in range(0, dropped.shape[dim], size):
            part = dropped.narrow(dim, s0, min(size, dropped.shape[dim] - s0))
            assert _within_binomial(part.sum().item(), part.numel(), P), (dim, s0)
    # the same seed gives the same mask, another seed another one
    again = _attention_probs(qkv, B, N, heads, dh, pad, (P, 1234))
    assert torch.equal(again, got)
    other = _attention_probs(qkv, B, N, heads, dh, pad, (P, 1235)) == 0
    assert (other != dropped).float().mean().item() > 0.5 * 2 * P * (1 - P)


def test_attention_dropout_mask_depends_on_indices_only():
    """Two different inputs, one of them with steep rows that take the two-pass softmax, give the same mask."""
    B, heads, N, dh = 4, 12, 197, 64
    masks = []
    for steep in (False, True):
        qkv = _qkv(B, N, heads, dh, 0, seed=77, steep=steep)
        if steep:
            q, k = (qkv.float().view(B, N, 3, heads, dh).permute(2, 0, 3, 1, 4)[i] for i in range(2))
            s = q @ k.transpose(-1, -2) * dh ** -0.5
            assert ((s[:2].amax(-1) - s[:2, ..., :32].amax(-1)) * 1.4427 > 128).any()  # the two-pass case is present
        full = _attention_probs(qkv, B, N, heads, dh, 0, (0.0, 0))
        got = _attention_probs(qkv, B, N, heads, dh, 0, (P, 99))
        # near one-hot rows underflow to zeros or to bf16 subnormals, which keep too few bits to read a 1 / (1 - p)
        readable = full > 1e-30
        ratio = (got[readable & (got != 0)] / full[readable & (got != 0)] * (1 - P) - 1).abs().max().item()
        print(f"steep={steep}: {readable.float().mean().item():.3f} of the probabilities readable, kept / undropped "
              f"ratio off 1 / (1 - p) by at most {ratio:.2e}")
        assert ratio < 1e-2
        masks.append((got == 0, readable))
    both = masks[0][1] & masks[1][1]
    assert both.sum().item() > 0.5 * both.numel()
    assert torch.equal(masks[0][0][both], masks[1][0][both])
    rate = masks[1][0][masks[1][1]].float().mean().item()
    print(f"steep input: drop rate {rate:.5f} on the readable probabilities")
    assert _within_binomial(masks[1][0][masks[1][1]].sum().item(), masks[1][1].sum().item(), P)


def test_attention_dropout_p0_is_the_plain_kernel_and_mean_is_unbiased():
    B, heads, N, dh = 2, 4, 256, 128
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


# ---------------------------------------------------------------------- linear ----
def _lin_inputs(M, K, N, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    y = (torch.randn(M, K, generator=g) * 0.5).to(DEV).bfloat16()
    w = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(DEV).bfloat16()
    gamma = (0.1 * (1 + 0.1 * torch.randn(N, generator=g))).to(DEV)
    bias = (torch.randn(N, generator=g) * 0.1).to(DEV)
    x = torch.randn(M, N, generator=g).to(DEV)
    return y, w, gamma, bias, x


@pytest.mark.parametrize("M,K,N", [(1000, 512, 512), (256 * 2, 2048, 512), (300, 512, 1024)])
def test_linear_dropout_before_the_fp32_residual(M, K, N):
    """out = res + drop(gamma (W y + b)): dropped -> exactly res, kept -> res + (W y + b) gamma / (1 - p)."""
    y, w, gamma, bias, x = _lin_inputs(M, K, N, seed=M + N)
    kw = dict(scale=gamma, bias=gamma * bias, res=x, res_mode=2)
    out = nat.linear_f32(y, w, out_dtype=torch.float32, dropout=(P, 42), **kw)
    out_b = nat.linear_f32(y, w, out_dtype=torch.bfloat16, dropout=(P, 42), **kw)
    plain = nat.linear_f32(y, w, out_dtype=torch.float32, **kw)
    zero = nat.linear_f32(y, w, out_dtype=torch.float32, dropout=(0.0, 42), **kw)
    other = nat.linear_f32(y, w, out_dtype=torch.float32, dropout=(P, 43), **kw)
    again = nat.linear_f32(y, w, out_dtype=torch.float32, dropout=(P, 42), **kw)
    torch.cuda.synchronize()
    assert torch.equal(zero, plain)
    assert torch.equal(again, out)
    ref_y = (gamma.double() * (y.double() @ w.double().t() + bias.double()))
    expect = x.double() + ref_y / (1 - P)
    dropped = out == x
    assert _within_binomial(dropped.sum().item(), dropped.numel(), P)
    err32 = ((out.double() - expect).abs()[~dropped]).max().item() / expect.abs().max().item()
    assert err32 < 1e-5
    # bf16 output of the same launch shape and seed: the same mask
    assert torch.equal(out_b[dropped], x[dropped].bfloat16())
    errb = ((out_b.double() - expect).abs() / (expect.abs() + 1e-3))[~dropped].max().item()
    assert errb < 8e-3
    drop_other = other == x
    assert (drop_other != dropped).float().mean().item() > 0.5 * 2 * P * (1 - P)
    print(f"linear_mc fp32 residual ({M},{K},{N}): drop rate {dropped.float().mean().item():.5f}, worst kept error "
          f"fp32 {err32:.2e} (of max), bf16 {errb:.2e} (relative)")


def test_linear_dropout_after_gelu_and_one_decision_rule():
    """fc1 + GELU with a bf16 output (the MODE 3 epilogue): dropped -> 0, kept -> GELU / (1 - p).  The fp32-output
    epilogue without residual decides with the same Philox(seed; row * N + col) rule."""
    M, K, N = 1000, 512, 2048
    y, w, _, bias, _ = _lin_inputs(M, K, N, seed=3)
    plain = nat.linear(y, w, bias=bias, act=1)
    got = nat.linear(y, w, bias=bias, act=1, dropout=(P, 77))
    zero = nat.linear(y, w, bias=bias, act=1, dropout=(0.0, 77))
    f32 = nat.linear_f32(y, w, bias=bias, act=1, out_dtype=torch.float32, dropout=(P, 77))
    torch.cuda.synchronize()
    assert torch.equal(zero, plain)
    readable = plain != 0  # GELU of very negative inputs is exactly 0 either way
    dropped = (got == 0) & readable
    n = readable.sum().item()
    assert n > 0.99 * readable.numel()
    assert _within_binomial(dropped.sum().item(), n, P)
    kept = readable & ~dropped
    ref = plain.float() / (1 - P)
    err = ((got.float() - ref).abs() / (ref.abs() + 1e-2))[kept].max().item()
    assert err < 1e-2
    assert torch.equal(f32[readable] == 0, dropped[readable])
    print(f"linear_mc GELU bf16 ({M},{K},{N}): drop rate {dropped.sum().item() / n:.5f}, worst kept relative error "
          f"{err:.2e}")


# ----------------------------------------------------------------- model level ----
def _inputs(n=4):
    dwi_raw, dce_raw, _, _ = op.synthetic_raw(n, seed=22, kind="S")
    return dwi_raw / dwi_raw.amax(dim=(1, 2, 3), keepdim=True), dce_raw


def _oracle_passes(p, sds, dwi, dce, passes, **kw):
    torch.manual_seed(3)
    torch.set_num_threads(max(torch.get_num_threads(), 8))
    ref = []
    with torch.no_grad():
        for _ in range(passes):
            _, ad, md = mdo.encoder_forward(sds["dwi"], "dwi", p, dwi, **kw)
            _, ac, mc = mdo.encoder_forward(sds["dce"], "dce", p, dce, **kw)
            ref.append(torch.softmax(mo.fusion_forward(sds["fusion"], p, ad["raw_feats"], ac["raw_feats"], md, mc)[0], 1))
    return torch.stack(ref)


def _agrees(tag, mean_a, std_a, ref, passes):
    ref_mean, ref_std = ref.mean(0), ref.std(0)
    se = torch.sqrt(ref_std ** 2 + std_a.cpu() ** 2) / passes ** 0.5
    diff = (mean_a.cpu() - ref_mean).abs()
    ratio = (std_a.cpu().mean() / ref_std.mean()).item()
    print(f"{tag}: max |mean - oracle mean| {diff.max().item():.3e}, spread ratio {ratio:.3f}, "
          f"mean spread {std_a.mean().item():.3e}")
    assert (diff <= 5 * se + HYBRID_TOL * ref_mean.max()).all(), (diff, se)
    assert 0.6 < ratio < 1.6, ratio


def test_hybrid_mc_dropout_prediction_is_statistically_the_reference():
    """predict_mc_dropout with use_hybrid_transformer=True: the CNN blocks drop at the config's 0.2, the transformer's
    attention / proj / MLP dropouts at their own 0.1."""
    p, sds, mods = _build(hybrid=True)
    lm = _lightning(p, mods)
    n, passes = 4, 48
    dwi, dce = _inputs(n)
    eval_before = _run_product(mods, dwi, dce)[2][0]
    lm.set_mc_seed(5)
    mean_a, std_a, _ = lm.predict_mc_dropout(dwi.to(DEV), dce.to(DEV), passes=passes)
    lm.set_mc_seed(5)
    mean_b, _, _ = lm.predict_mc_dropout(dwi.to(DEV), dce.to(DEV), passes=passes)
    torch.cuda.synchronize()
    assert _relmax(mean_a, mean_b) <= 2e-3                      # same seed, same passes (up to fp32 atomics)
    assert std_a.max().item() > 1e-4
    for k in ("dwi", "dce"):
        assert not any(m.training for m in mods[k].modules())   # train flags restored
    eval_after = _run_product(mods, dwi, dce)[2][0]
    assert _relmax(eval_after, eval_before) <= 2e-3
    _agrees("hybrid MC dropout, all dropouts", mean_a, std_a, _oracle_passes(p, sds, dwi, dce, passes, mc_dropout=True),
            passes)
    mean_t, _, _ = lm.predict_tta_mc(dwi.to(DEV), dce.to(DEV), passes=4)
    assert mean_t.shape == (n, 4) and torch.isfinite(mean_t).all() and abs(mean_t.sum(1).mean().item() - 1) < 1e-3


def test_hybrid_mc_dropout_transformer_only_with_blocks_at_p0():
    """Blocks built with dropout = 0 (their Dropouts in train mode at p = 0): only the transformer drops, and the
    convolutions must not pick up the transformer's p."""
    p, sds, mods = _build(hybrid=True)
    for k in ("dwi", "dce"):
        p[f"{k}_model_parameters"]["dropout"] = 0.0
        for blk in (mods[k].block1, mods[k].block2):
            for m in blk.modules():
                if isinstance(m, torch.nn.Dropout):
                    m.p = 0.0
    lm = _lightning(p, mods)
    passes = 48
    dwi, dce = _inputs()
    lm.set_mc_seed(8)
    mean_a, std_a, _ = lm.predict_mc_dropout(dwi.to(DEV), dce.to(DEV), passes=passes)
    torch.cuda.synchronize()
    assert std_a.max().item() > 1e-4
    _agrees("hybrid MC dropout, transformer only", mean_a, std_a,
            _oracle_passes(p, sds, dwi, dce, passes, mc_dropout=True), passes)


def test_hybrid_mc_dropout_cnn_blocks_only():
    """Only the CNN blocks' Dropouts in train mode: the transformer stage runs its eval launches."""
    p, sds, mods = _build(hybrid=True)
    passes = 48
    dwi, dce = _inputs()
    for k, seed in (("dwi", 11), ("dce", 12)):
        mods[k].set_mc_seed(seed)
        for blk in (mods[k].block1, mods[k].block2):
            for m in blk.modules():
                if isinstance(m, torch.nn.Dropout):
                    m.train()
    probs = []
    with torch.no_grad():
        for _ in range(passes):
            probs.append(torch.softmax(_run_product(mods, dwi, dce)[2][0], 1))
    for k in ("dwi", "dce"):
        mods[k].eval()
    probs = torch.stack(probs)
    assert probs.std(0).max().item() > 1e-4
    _agrees("hybrid MC dropout, CNN blocks only", probs.mean(0), probs.std(0),
            _oracle_passes(p, sds, dwi, dce, passes, mc_dropout=True, transformer_dropout=False), passes)
